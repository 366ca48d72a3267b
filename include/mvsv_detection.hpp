// mvsv_detection.hpp -- the disparity consumers right after the hot path (SURVEY.md 8f rows f1, f2), as host C++
// on top of the engine's outputs: the per-ROI means come from MVSV_STAGE_MEANS, the min/max disparity from
// mvsv_download_minmax, so no pass over the disparity map is left on the CPU.
//
// Mirrors (same names, argument meaning, quirks) of the reference's
//   Utility::calcCoordinate / calcDistance / calcDMapValues   src/utility.cpp:176-240
//   struct Subimage / struct Samplepoint                       inc/Subimage.h, inc/Samplepoint.h
//   MeanDisparityDetection::{init,build,detectObstacles}       src/MeanDisparityDetection.cpp:71-266
//   SamplepointDetection::{init,build,detectObstacles}         src/SamplePointDetection.cpp:29-178
//   ply::write (PLAIN / WITH_COLOR)                            src/ply.cpp:36-95
// Differences, all deliberate: build() takes the means computed on the GPU instead of a cv::Mat; detectObstacles()
// returns the found points and leaves writing the PLY file to the caller (`ply::write`), the reference hard-codes
// "pcl/subimage_detection/pcl_NNNN.ply"; Q is a row-major float[16] instead of a CV_32F cv::Mat.
#pragma once
#include <cmath>
#include <fstream>
#include <ostream>
#include <string>
#include <utility>
#include <vector>

namespace mvsv {

struct Point { int x, y; };
struct Vec4 { float v[4]; };

// reference inc/utility.h:49-54
struct dMapValues { float dValue, image_x, image_y; };

namespace Utility {

// src/utility.cpp:176-200: d = dValue/16; c = Q*[x,y,d,1]^T; c /= c[3]; z := 0 if z/1000 is infinite.
// cv::Mat_<float> products accumulate in double; `c /= c(3)` multiplies by the double reciprocal.
inline Vec4 calcCoordinate(dMapValues m, const float* Q)
{
    const float in[4] = {m.image_x, m.image_y, m.dValue / 16, 1.f};
    float c[4];
    for (int r = 0; r < 4; ++r) {
        double acc = 0;
        for (int k = 0; k < 4; ++k) acc += (double)Q[r * 4 + k] * (double)in[k];
        c[r] = (float)acc;
    }
    const double inv = 1.0 / (double)c[3];
    Vec4 out;
    for (int r = 0; r < 4; ++r) out.v[r] = (float)(c[r] * inv);
    const float distance = out.v[2] / 1000;
    if (std::isinf(distance)) out.v[2] = 0;
    return out;
}

// src/utility.cpp:202-222
inline float calcDistance(dMapValues m, const float* Q, int /*binning*/)
{
    const float in[4] = {m.image_x, m.image_y, m.dValue / 16, 1.f};
    double z = 0, w = 0;
    for (int k = 0; k < 4; ++k) { z += (double)Q[2 * 4 + k] * in[k]; w += (double)Q[3 * 4 + k] * in[k]; }
    const float zz = (float)((float)z * (1.0 / (double)(float)w));
    const float distance = zz / 1000;
    return std::isinf(distance) ? 0.f : distance;
}

// src/utility.cpp:224-240
inline dMapValues calcDMapValues(const float c[3], const float* Q)
{
    const float numerator = Q[2 * 4 + 3] - c[2] * Q[3 * 4 + 3];
    const float denominator = c[2] * Q[3 * 4 + 2];
    const float disparity_value = numerator / denominator;
    dMapValues r;
    r.image_x = c[0] * (disparity_value * Q[3 * 4 + 2] * Q[3 * 4 + 3]) + Q[0 * 4 + 3];
    r.image_y = c[1] * (disparity_value * Q[3 * 4 + 2] * Q[3 * 4 + 3]) + Q[1 * 4 + 3];
    r.dValue = disparity_value * 16;
    return r;
}

}  // namespace Utility

// inc/Subimage.h
struct Subimage {
    Point tl{0, 0}, br{0, 0}, roi_center{0, 0};
    float value = 0;
    Subimage() {}
    Subimage(Point tl_, Point br_) : tl(tl_), br(br_)
    {
        roi_center = Point{tl.x + (br.x - tl.x) / 2, tl.y + (br.y - tl.y) / 2};
    }
};

// inc/Samplepoint.h (roi = [center - radius, center + radius + 1) in both axes)
struct Samplepoint {
    Point center{0, 0};
    int radius = 0;
    int roi[4] = {0, 0, 0, 0};   // x, y, w, h
    float value = 0;
    Samplepoint() {}
    Samplepoint(Point c, int r) : center(c), radius(r)
    {
        roi[0] = c.x - r; roi[1] = c.y - r; roi[2] = 2 * r + 1; roi[3] = 2 * r + 1;
    }
};

// pixelShift of createDMapROIS (trgt/demo.cpp:87-101): the consumers see dMapRaw(cols >= pixelShift).  numDisp / 2,
// made even; the reference's adjustment for an odd half (`shift + (cols - shift % 8)`, operator precedence as written)
// is kept as is.  Pass the result as x_offset to the detectors' init().
inline int dMapRoiOffset(int numDisp, int cols)
{
    int pixelShift = numDisp / 2;
    if (pixelShift % 2 == 1) {
        pixelShift = pixelShift + 1;
        if ((cols - pixelShift) % 8 != 0) pixelShift = pixelShift + (cols - pixelShift % 8);
    }
    return pixelShift;
}

// src/ObstacleDetection.cpp + inc/ObstacleDetection.h
class ObstacleDetection {
public:
    enum MODE { MEAN_DISTANCE, SAMPLEPOINTS };
    virtual ~ObstacleDetection() {}
    virtual void build(const float* means, int binning, int mode) = 0;
    virtual void detectObstacles() = 0;
    std::pair<float, float> getRange() const { return mRange; }
    void setRange(std::pair<float, float> const& r) { mRange = r; }
    std::pair<float, float> getRangeDisparity() const { return mRangeDisparity; }
    // ROIs (x, y, w, h in RAW disparity-map coordinates) to hand to mvsv_set_mean_rois, in build() order
    const std::vector<int>& rois() const { return mRois; }
    const std::vector<Vec4>& getFoundPoints() const { return mFoundPoints; }

protected:
    void initRangeDisparity(const float* Q, float min_distance, float max_distance)
    {
        for (int i = 0; i < 16; ++i) mQ[i] = Q[i];
        const float lower[3] = {0, 0, min_distance * 1000}, upper[3] = {0, 0, max_distance * 1000};
        mRangeDisparity = std::make_pair(Utility::calcDMapValues(lower, mQ).dValue, Utility::calcDMapValues(upper, mQ).dValue);
    }
    std::pair<float, float> mRange{0.f, 0.f}, mRangeDisparity{0.f, 0.f};
    float mQ[16];
    std::vector<int> mRois;
    std::vector<Vec4> mFoundPoints;
};

// src/MeanDisparityDetection.cpp
class MeanDisparityDetection : public ObstacleDetection {
public:
    enum MODE { MEAN_DISTANCE, MEAN_VALUE };
    // reference: init(cv::Mat const& reference, Q, min, max); `reference` is the dMapWork view, i.e. the raw map
    // without its first x_offset columns (trgt/demo.cpp:87-113,236-237) -- only its size is used.
    void init(int cols, int rows, const float* Q, float min_distance, float max_distance, int x_offset = 0)
    {
        mSubimageVec.clear();
        mRois.clear();
        const int distanceX = cols / 9, distanceY = rows / 9;
        for (int r = 0; r < 9; ++r)
            for (int c = 0; c < 9; ++c) {
                const Point tl{c * distanceX, r * distanceY}, br{c * distanceX + distanceX, r * distanceY + distanceY};
                mSubimageVec.push_back(Subimage(tl, br));
                mFoundObstacles.push_back(Subimage(tl, br));       // sic: the reference pre-fills the found list too
                mRois.push_back(x_offset + tl.x); mRois.push_back(tl.y); mRois.push_back(distanceX); mRois.push_back(distanceY);
            }
        initRangeDisparity(Q, min_distance, max_distance);
    }
    std::vector<Subimage> getSubimageVec() const { return mSubimageVec; }
    std::vector<float> getMeanMap() const { return mMeanMap; }
    std::vector<float> getMeanDistanceMap() const { return mMeanDistanceMap; }
    std::vector<Subimage> getFoundObstacles() const { return mFoundObstacles; }
    int getObstacleCounter() const { return mObstacleCounter; }
    int getDetectionMode() const { return mDetectionMode; }

    // means[i] = Utility::calcMeanDisparity of Subimage i (MVSV_STAGE_MEANS output, same order as rois())
    void build(const float* means, int /*binning*/, int mode) override
    {
        switch (mode) {
            case MEAN_DISTANCE: {
                mDetectionMode = MEAN_DISTANCE;
                mMeanDistanceMap.clear();
                for (size_t i = 0; i < mSubimageVec.size(); ++i) {
                    dMapValues m;
                    m.image_x = (float)mSubimageVec[i].roi_center.x; m.image_y = (float)mSubimageVec[i].roi_center.y;
                    m.dValue = means[i];
                    mMeanDistanceMap.push_back(Utility::calcDistance(m, mQ, 0));
                }
            }
            // no break: the reference falls through into MEAN_VALUE (src/MeanDisparityDetection.cpp:191-193)
            case MEAN_VALUE: {
                mDetectionMode = MEAN_VALUE;
                mMeanMap.clear();
                for (size_t i = 0; i < mSubimageVec.size(); ++i) {
                    mSubimageVec[i].value = means[i];
                    mMeanMap.push_back(means[i]);
                }
            }
        }
    }

    void detectObstacles() override
    {
        if (mDetectionMode == MEAN_DISTANCE) return;    // unreachable after build() (fall-through), kept for fidelity
        mFoundObstacles.clear();
        mFoundPoints.clear();
        for (size_t i = 0; i < mMeanMap.size(); ++i) {
            if (mMeanMap[i] < mRangeDisparity.first && mMeanMap[i] > mRangeDisparity.second) {
                const Subimage s = mSubimageVec[i];
                mFoundObstacles.push_back(s);
                dMapValues m;
                m.image_x = (float)s.roi_center.x; m.image_y = (float)s.roi_center.y; m.dValue = mMeanMap[i];
                mFoundPoints.push_back(Utility::calcCoordinate(m, mQ));
            }
        }
        if (!mFoundPoints.empty()) ++mObstacleCounter;   // the reference writes pcl_NNNN.ply here
    }

private:
    std::vector<Subimage> mSubimageVec, mFoundObstacles;
    std::vector<float> mMeanMap, mMeanDistanceMap;
    int mDetectionMode = MEAN_VALUE, mObstacleCounter = 0;
};

// src/SamplePointDetection.cpp
class SamplepointDetection : public ObstacleDetection {
public:
    void init(int cols, int rows, const float* Q, float min_distance, float max_distance, int x_offset = 0)
    {
        mSPVec.clear();
        mRois.clear();
        const int distanceX = cols / 8, distanceY = rows / 8;
        for (int c = 1; c < distanceX; ++c)
            for (int r = 1; r < distanceY; ++r) {
                const Samplepoint sp(Point{c * (cols / distanceX), r * (rows / distanceY)}, 2);
                mSPVec.push_back(sp);
                mFoundObstacles.push_back(sp);
                mRois.push_back(x_offset + sp.roi[0]); mRois.push_back(sp.roi[1]); mRois.push_back(sp.roi[2]); mRois.push_back(sp.roi[3]);
            }
        initRangeDisparity(Q, min_distance, max_distance);
    }
    std::vector<Samplepoint> getSamplepointVec() const { return mSPVec; }
    std::vector<Samplepoint> getFoundObstacles() const { return mFoundObstacles; }
    int getObstacleCounter() const { return mObstacleCounter; }

    void build(const float* means, int /*binning*/, int /*mode*/) override
    {
        mDistanceVec.clear();
        for (size_t i = 0; i < mSPVec.size(); ++i) { mSPVec[i].value = means[i]; mDistanceVec.push_back(means[i]); }
    }

    void detectObstacles() override
    {
        mFoundObstacles.clear();
        mFoundPoints.clear();
        for (size_t i = 0; i < mDistanceVec.size(); ++i) {
            if (mDistanceVec[i] < mRangeDisparity.first && mDistanceVec[i] > mRangeDisparity.second) {
                Samplepoint s = mSPVec[i];
                s.value = mDistanceVec[i];
                mFoundObstacles.push_back(s);
                dMapValues m;
                m.image_x = (float)s.center.x; m.image_y = (float)s.center.y; m.dValue = mDistanceVec[i];
                mFoundPoints.push_back(Utility::calcCoordinate(m, mQ));
            }
        }
        if (!mFoundPoints.empty()) ++mObstacleCounter;
    }

private:
    std::vector<Samplepoint> mSPVec, mFoundObstacles;
    std::vector<float> mDistanceVec;
    int mObstacleCounter = 0;
};

// src/ply.cpp: ASCII PLY; WITH_COLOR greys every vertex by (z - min)/(max - min)*255 with min/max the smallest and
// largest positive DISPARITY value of the map (Utility::calcMinMaxDisparity, src/utility.cpp:287-304) -- the
// reference mixes millimetres and disparity units there; reproduced as is.  minmax comes from mvsv_download_minmax; a
// whole map's points (Utility::dmap2pcl, src/utility.cpp:242-262) from MVSV_STAGE_POINTS and mvsv_download_points.
class ply {
public:
    enum MODE { PLAIN, WITH_COLOR, WITH_COLOR_SHADING };
    ply(std::string const& author, std::string const& object_name) : mAuthor(author), mObjectName(object_name) {}
    ply(std::string const& author, std::string const& object_name, short minDisp, short maxDisp)
        : mAuthor(author), mObjectName(object_name), mHaveMap(true), mMin(minDisp), mMax(maxDisp) {}

    bool write(std::ostream& out, std::vector<Vec4> const& to_write, int mode) const
    {
        return write_n(out, to_write.size(), [&](size_t i) { return to_write[i].v; }, mode);
    }
    bool write(std::string const& filename, std::vector<Vec4> const& to_write, int mode) const
    {
        if (mode != PLAIN && !mHaveMap) return false;
        std::ofstream f(filename.c_str());
        return f.is_open() && write(f, to_write, mode);
    }
    // n points of x, y, z floats one after the other: the layout mvsv_download_points writes, so that the point list of
    // a whole map (Utility::dmap2pcl) goes to the file without a copy into Vec4.  The same bytes as the Vec4 overload.
    bool write(std::ostream& out, const float* xyz, size_t n, int mode) const
    {
        return write_n(out, n, [&](size_t i) { return xyz + 3 * i; }, mode);
    }
    bool write(std::string const& filename, const float* xyz, size_t n, int mode) const
    {
        if (mode != PLAIN && !mHaveMap) return false;
        std::ofstream f(filename.c_str());
        return f.is_open() && write(f, xyz, n, mode);
    }

private:
    // at(i): the x, y, z of vertex i
    template <class At>
    bool write_n(std::ostream& out, size_t n, At at, int mode) const
    {
        if (mode != PLAIN && !mHaveMap) return false;
        out << "ply\nformat ascii 1.0\ncomment author: " << mAuthor << "\ncomment object:" << mObjectName << "\n";
        out << "element vertex " << std::to_string(n) << "\n";
        out << "property float x\nproperty float y\nproperty float z\n";
        if (mode != PLAIN) out << "property uchar red\nproperty uchar green\nproperty uchar blue\n";
        out << "end_header\n";
        for (size_t i = 0; i < n; ++i) {
            const float* t = at(i);
            out << t[0] << " " << t[1] << " " << t[2];
            if (mode == WITH_COLOR) {
                const int g = int((t[2] - mMin) / (mMax - mMin) * 255.0);
                out << " " << g << " " << g << " " << g;
            }
            out << "\n";
        }
        return true;
    }

    std::string mAuthor, mObjectName;
    bool mHaveMap = false;
    short mMin = 0, mMax = 0;
};

}  // namespace mvsv
