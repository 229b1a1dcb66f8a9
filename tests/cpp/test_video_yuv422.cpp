// C++ check of processFramesInMemory (csrc/videoprocessingcontext.hpp) on packed YUYV frames, the form a V4L2 webcam hands over: the same
// clip on ONE Watermark object and on TWO (contiguous chunks of the global frame index, one host thread each) must agree, which needs the
// 2 bytes per pixel in the per-chunk output offsets.
// usage: test_video_yuv422 <w.dat> <rows> <cols> <frames.u8> <nframes> <linesize> <interval> <out.u8>
// prints one line per result: "<name> <value>"; writes the one-object EMBED output (dense YUYV frames) to <out.u8>.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <vector>

#include "videoprocessingcontext.hpp"

int main(int argc, char** argv)
{
    if (argc != 9) { std::cerr << "usage\n"; return 2; }
    const int rows = atoi(argv[2]), cols = atoi(argv[3]), nframes = atoi(argv[5]), linesize = atoi(argv[6]), interval = atoi(argv[7]);
    std::vector<unsigned char> frames((size_t)nframes * rows * linesize);
    {
        std::ifstream f(argv[4], std::ios::binary);
        if (!f.read(reinterpret_cast<char*>(frames.data()), (std::streamsize)frames.size())) { std::cerr << "cannot read " << argv[4] << "\n"; return 2; }
    }
    try {
        Watermark one(rows, cols, argv[1], 3, 40.0f);
        const Watermark second(one);
        const size_t obytes = (size_t)nframes * rows * 2 * cols;
        std::vector<unsigned char> out1(obytes), out2(obytes, 0x5A);
        std::vector<float> a1((size_t)nframes), a2((size_t)nframes), c1((size_t)nframes), c2((size_t)nframes);
        const int64_t n1 = processFramesInMemory({&one}, rows, cols, interval, linesize, WM_VIDEO_EMBED, frames.data(), out1.data(), 0, nframes,
                                                 a1.data(), WM_PACKED_YUYV);
        const int64_t n2 = processFramesInMemory({&one, &second}, rows, cols, interval, linesize, WM_VIDEO_EMBED, frames.data(), out2.data(), 0,
                                                 nframes, a2.data(), WM_PACKED_YUYV);
        // detection of the watermarked frames: dense rows of 2 * cols bytes
        processFramesInMemory({&one}, rows, cols, interval, 2 * cols, WM_VIDEO_DETECT, out1.data(), nullptr, 0, nframes, c1.data(), WM_PACKED_YUYV);
        processFramesInMemory({&one, &second}, rows, cols, interval, 2 * cols, WM_VIDEO_DETECT, out2.data(), nullptr, 0, nframes, c2.data(),
                              WM_PACKED_YUYV);
        std::printf("frames %lld %lld\n", (long long)n1, (long long)n2);
        std::printf("equal_pixels %d\n", (int)(out1 == out2));
        int a_equal = 1, nan_ok = 1;
        double corr_rel = 0.0;
        for (int i = 0; i < nframes; i++) {
            const bool gated = i % interval == 0;
            if (std::memcmp(&a1[(size_t)i], &a2[(size_t)i], sizeof(float)) != 0) a_equal = 0;
            if (std::isnan(a1[(size_t)i]) == gated || std::isnan(c1[(size_t)i]) == gated || std::isnan(c2[(size_t)i]) == gated) nan_ok = 0;
            if (gated) corr_rel = std::max(corr_rel, std::fabs((double)c1[(size_t)i] - c2[(size_t)i]) / std::fabs((double)c1[(size_t)i]));
            std::printf("a_%d %.9g\ncorr_%d %.9g\n", i, a1[(size_t)i], i, c1[(size_t)i]);
        }
        std::printf("equal_a %d\nnan_where_gated_off %d\ncorr_max_rel %.9g\n", a_equal, nan_ok, corr_rel);
        std::ofstream f(argv[8], std::ios::binary);
        f.write(reinterpret_cast<const char*>(out1.data()), (std::streamsize)out1.size());
    } catch (const std::exception& e) {
        std::cerr << "exception: " << e.what();
        return 1;
    }
    return 0;
}
