// The found-obstacle records of MVSV_STAGE_DETECT as include/mvsv_detection.hpp defines them, frame by frame: both
// reference detectors (MeanDisparityDetection detector 0, SamplepointDetection detector 1, ROIs in that order) run
// build() + detectObstacles() on each frame's means with that frame's Q.
// usage: detect_records <cols> <rows> <x_offset> <min0> <max0> <min1> <max1> <qs.bin> <means.bin> [<offsets.bin> <records.bin>]
//   qs.bin: 16 f32 per frame; means.bin: the ROI means of every frame (81 sub-image means, then the sample points).
// prints
//   T <detector> <image_x> <image_y>            the table of mvsv_set_detection (detectionTable), one line per ROI
//   D <min0> <max0> <min1> <max1>               its distances
//   F <frame> <records> <counter0> <counter1>   then one line per record, in ROI order:
//   R <roi> <value> <x> <y> <z> <w>             floats as %a
//   B <frame> <0|1>                             buildFromObstacles() on the frame's records gives what detectObstacles()
//                                               gave (found lists, points bit for bit, counters); the records are those of
//                                               offsets.bin / records.bin when given (a device download), else the above
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <utility>
#include <vector>
#include "mvsv_detection.hpp"

template <class T>
static std::vector<T> slurp(const char* fn)
{
    std::vector<T> v;
    FILE* f = std::fopen(fn, "rb");
    if (!f) return v;
    T x;
    while (std::fread(&x, sizeof(T), 1, f) == 1) v.push_back(x);
    std::fclose(f);
    return v;
}

static bool same_points(const std::vector<mvsv::Vec4>& a, const std::vector<mvsv::Vec4>& b)
{
    return a.size() == b.size() && (a.empty() || std::memcmp(a.data(), b.data(), a.size() * sizeof(mvsv::Vec4)) == 0);
}

int main(int argc, char** argv)
{
    if (argc != 10 && argc != 12) return 2;
    const int cols = std::atoi(argv[1]), rows = std::atoi(argv[2]), xoff = std::atoi(argv[3]);
    const float dist[4] = {(float)std::atof(argv[4]), (float)std::atof(argv[5]), (float)std::atof(argv[6]), (float)std::atof(argv[7])};
    const std::vector<float> qs = slurp<float>(argv[8]), means = slurp<float>(argv[9]);
    const int nf = (int)qs.size() / 16;
    mvsv::MeanDisparityDetection m, m2;
    mvsv::SamplepointDetection sd, sd2;
    m.init(cols, rows, qs.data(), dist[0], dist[1], xoff);
    sd.init(cols, rows, qs.data(), dist[2], dist[3], xoff);
    std::vector<int> det;
    std::vector<float> centers, ranges;
    mvsv::detectionTable(m, det, centers, ranges);
    mvsv::detectionTable(sd, det, centers, ranges);
    const int nm = (int)m.rois().size() / 4, n = (int)det.size();
    if (means.size() != (size_t)nf * n) { std::fprintf(stderr, "means size\n"); return 4; }
    for (int i = 0; i < n; ++i) std::printf("T %d %.9g %.9g\n", det[i], centers[2 * i], centers[2 * i + 1]);
    std::printf("D %.9g %.9g %.9g %.9g\n", ranges[0], ranges[1], ranges[2], ranges[3]);
    // ROI index of a found Subimage (by its top-left corner) and of a found Samplepoint (by its center)
    std::map<std::pair<int, int>, int> m_index, sd_index;
    for (int i = 0; i < nm; ++i) m_index[{m.getSubimageVec()[i].tl.x, m.getSubimageVec()[i].tl.y}] = i;
    for (int i = 0; i < n - nm; ++i) sd_index[{sd.getSamplepointVec()[i].center.x, sd.getSamplepointVec()[i].center.y}] = nm + i;

    std::vector<long long> dev_offs;
    std::vector<mvsv_obstacle> dev_rec;
    if (argc == 12) {
        dev_offs = slurp<long long>(argv[10]);
        dev_rec = slurp<mvsv_obstacle>(argv[11]);
        if ((int)dev_offs.size() != nf + 1 || (long long)dev_rec.size() < dev_offs[nf]) { std::fprintf(stderr, "records size\n"); return 5; }
    }
    for (int f = 0; f < nf; ++f) {
        const float* Q = qs.data() + 16 * f;
        // init() per frame: the frame's Q gives its ranges (several rigs); the counters live on in m2 / sd2 only
        m.init(cols, rows, Q, dist[0], dist[1], xoff);
        sd.init(cols, rows, Q, dist[2], dist[3], xoff);
        m2.init(cols, rows, Q, dist[0], dist[1], xoff);
        sd2.init(cols, rows, Q, dist[2], dist[3], xoff);
        const float* fm = means.data() + (size_t)f * n;
        m.build(fm, 0, mvsv::MeanDisparityDetection::MEAN_VALUE);
        m.detectObstacles();
        sd.build(fm + nm, 0, 0);
        sd.detectObstacles();
        std::vector<mvsv_obstacle> rec;
        const std::vector<mvsv::Subimage> fM = m.getFoundObstacles();
        const std::vector<mvsv::Samplepoint> fS = sd.getFoundObstacles();
        for (size_t k = 0; k < fM.size(); ++k) {
            mvsv_obstacle o;
            o.roi = m_index.at({fM[k].tl.x, fM[k].tl.y});
            o.value = fM[k].value;
            std::memcpy(o.xyzw, m.getFoundPoints()[k].v, sizeof(o.xyzw));
            rec.push_back(o);
        }
        for (size_t k = 0; k < fS.size(); ++k) {
            mvsv_obstacle o;
            o.roi = sd_index.at({fS[k].center.x, fS[k].center.y});
            o.value = fS[k].value;
            std::memcpy(o.xyzw, sd.getFoundPoints()[k].v, sizeof(o.xyzw));
            rec.push_back(o);
        }
        std::printf("F %d %zu %d %d\n", f, rec.size(), m.getObstacleCounter(), sd.getObstacleCounter());
        for (const mvsv_obstacle& o : rec)
            std::printf("R %d %a %a %a %a %a\n", o.roi, o.value, o.xyzw[0], o.xyzw[1], o.xyzw[2], o.xyzw[3]);
        const mvsv_obstacle* r = argc == 12 ? dev_rec.data() + dev_offs[f] : rec.data();
        const size_t cnt = argc == 12 ? (size_t)(dev_offs[f + 1] - dev_offs[f]) : rec.size();
        m2.buildFromObstacles(r, cnt, 0);
        sd2.buildFromObstacles(r, cnt, nm);
        bool same = same_points(m2.getFoundPoints(), m.getFoundPoints()) && same_points(sd2.getFoundPoints(), sd.getFoundPoints()) &&
                    m2.getObstacleCounter() == m.getObstacleCounter() && sd2.getObstacleCounter() == sd.getObstacleCounter();
        const std::vector<mvsv::Subimage> gM = m2.getFoundObstacles();
        const std::vector<mvsv::Samplepoint> gS = sd2.getFoundObstacles();
        same = same && gM.size() == fM.size() && gS.size() == fS.size();
        for (size_t k = 0; same && k < gM.size(); ++k)
            same = gM[k].tl.x == fM[k].tl.x && gM[k].tl.y == fM[k].tl.y && std::memcmp(&gM[k].value, &fM[k].value, 4) == 0;
        for (size_t k = 0; same && k < gS.size(); ++k)
            same = gS[k].center.x == fS[k].center.x && gS[k].center.y == fS[k].center.y && std::memcmp(&gS[k].value, &fS[k].value, 4) == 0;
        std::printf("B %d %d\n", f, same ? 1 : 0);
    }
    return 0;
}
