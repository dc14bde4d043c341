// lm_files.hpp — minimal raw containers that stand in for the reference's on-disk formats (AVI video,
// PNG background, OpenCV-YAML model / calibration: LocoMouse_class.cpp:367-463, 3095-3162).  Decoding
// and OpenCV-YAML parsing are outside the hot path (SURVEY §8f-3); these little-endian containers carry
// exactly the arrays those loaders would produce, so the class mirror can be driven end to end.
//   video        "LMV1" i32 n_frames, rows, cols        then n*rows*cols u8      (channel 0 of each frame)
//                       (read in frame ranges by lmmedia::index_lmv + read_frames, lm_media.hpp)
//   background   "LMI1" i32 rows, cols                  then rows*cols u8
//   model        "LMM1" 6 x { i32 rows, cols; f64 rho; rows*cols f32 }  in the order
//                       paw_bottom, snout_bottom, tail_bottom, paw_side, snout_side, tail_side
//   calibration  "LMC1" i32 n_rows, n_cols; i32 view_boxes[2][4] (side, bottom: x, y, w, h)
//                       then n_rows*n_cols i32 ind_warp_mapping (0-based raw-frame index)
//   boxes        "LMB1" i32 n  then u32 bb_x[n], bb_y_side[n], bb_y_bottom[n]   (pass-1 output)
//   results      "LMO1" written by LocoMouse::exportResults, see LocoMouse_class.cpp
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

namespace lmfile {

class Reader {
    FILE *f_ = nullptr;
    std::string name_;

public:
    Reader(const std::string &name, const char magic[4]) : name_(name) {
        f_ = std::fopen(name.c_str(), "rb");
        if (!f_) throw std::runtime_error("Cannot open file: " + name);
        char m[4];
        if (std::fread(m, 1, 4, f_) != 4 || std::memcmp(m, magic, 4) != 0) {
            std::fclose(f_);
            f_ = nullptr;
            throw std::runtime_error("Unexpected file format (" + std::string(magic, 4) + " expected): " + name);
        }
    }
    ~Reader() {
        if (f_) std::fclose(f_);
    }
    Reader(const Reader &) = delete;
    template <typename T>
    void read(T *dst, size_t count) {
        if (count && std::fread(dst, sizeof(T), count, f_) != count) throw std::runtime_error("File is truncated: " + name_);
    }
    int32_t i32() {
        int32_t v;
        read(&v, 1);
        return v;
    }
    double f64() {
        double v;
        read(&v, 1);
        return v;
    }
};

class Writer {
    FILE *f_ = nullptr;
    std::string name_;

public:
    Writer(const std::string &name, const char magic[4]) : name_(name) {
        f_ = std::fopen(name.c_str(), "wb");
        if (!f_) throw std::runtime_error("Cannot open output file: " + name);
        std::fwrite(magic, 1, 4, f_);
    }
    ~Writer() {
        if (f_) std::fclose(f_);
    }
    Writer(const Writer &) = delete;
    template <typename T>
    void write(const T *src, size_t count) {
        if (count && std::fwrite(src, sizeof(T), count, f_) != count) throw std::runtime_error("Write failed: " + name_);
    }
    void i32(int32_t v) { write(&v, 1); }
    void f64(double v) { write(&v, 1); }
};

}  // namespace lmfile
