// Writes one point list through both ply::write overloads of include/mvsv_detection.hpp: the std::vector<Vec4> one
// and the packed x, y, z floats of mvsv_download_points.  tests/test_points.py compares the two files byte for byte.
// usage: ply_points <xyz.bin (n x 3 f32)> <minDisp> <maxDisp> <mode> <out_vec4.ply> <out_packed.ply>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "mvsv_detection.hpp"

int main(int argc, char** argv)
{
    if (argc != 7) return 2;
    std::vector<float> xyz;
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) return 3;
    float v;
    while (std::fread(&v, 4, 1, f) == 1) xyz.push_back(v);
    std::fclose(f);
    if (xyz.size() % 3) return 4;
    const size_t n = xyz.size() / 3;
    std::vector<mvsv::Vec4> pts(n);
    for (size_t i = 0; i < n; ++i) {
        for (int k = 0; k < 3; ++k) pts[i].v[k] = xyz[3 * i + k];
        pts[i].v[3] = 1.f;
    }
    const mvsv::ply writer("Hagen Hiller", "pointcloud", (short)std::atoi(argv[2]), (short)std::atoi(argv[3]));
    const int mode = std::atoi(argv[4]);
    if (!writer.write(std::string(argv[5]), pts, mode)) return 5;
    if (!writer.write(std::string(argv[6]), xyz.data(), n, mode)) return 6;
    return 0;
}
