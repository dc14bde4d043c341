// lm_containers.hpp — the Matroska and QuickTime / MP4 indexers of lm_media.hpp.  Each makes one walk over the file's structure
// and fills an lmmedia::Index as index_avi does: the file offset and size of every frame's coded payload, or a RawChunk for
// every uncompressed frame.  read_frames, plan_windows, the reader thread and the device decoders work from that Index alone.
//   Matroska: the first video track (as OpenCV takes it), its frames from SimpleBlock and BlockGroup / Block in file order;
//     V_FFV1 (record = CodecPrivate), V_MS/VFW/FOURCC (CodecPrivate = BITMAPINFOHEADER: 'MPNG' / 'png ', 'FFV1', 'Y800' and
//     BI_RGB 24 / 32, top-down), V_UNCOMPRESSED (ColourSpace 'Y800' / 'GREY' / 'Y8  ', 'BGR' 24, 'RGB' 24).  Elements of unknown size (Segment,
//     Cluster) are walked through.  Matroska stores no frame count: OpenCV estimates one from the duration and the frame rate
//     (mkv_frame_count), and a file where that estimate differs from the frames found is refused.
//   QuickTime / MP4: the first 'vide' track; sample offsets from stsc + stco / co64, sizes from stsz; sample entries 'png ' /
//     'MPNG', 'FFV1' (record in the entry's 'glbl' box), 'raw ' (8-bit grey, inverted as libavformat reads it, and 24-bit RGB) and 'mp4v' whose esds object type
//     is PNG (0x6D).  'moov' may come before or after 'mdat'.
// Refused with the file name and the reason: laced blocks, encrypted or compressed tracks (ContentEncoding), fragmented MP4,
// edit lists other than the identity, non-zero composition offsets, truncated elements or boxes, and codecs this library
// does not decode.
#pragma once
#include <cmath>
#include <cstdint>
#include <string>
#include <vector>

#include "lm_media.hpp"

namespace lmmedia {
namespace detail {

inline uint64_t be_n(const uint8_t *p, size_t n) {
    uint64_t v = 0;
    for (size_t i = 0; i < n; ++i) v = (v << 8) | p[i];
    return v;
}
inline std::string fourcc_text(const uint8_t *p) {
    std::string s;
    for (int i = 0; i < 4; ++i) s += (p[i] >= 32 && p[i] < 127) ? (char)p[i] : '?';
    return s;
}

// Row stride of an uncompressed frame of `size` bytes, as libavcodec's raw decoder takes it and index_avi does: rows padded to
// 4 bytes when the frame holds that many, else tight; 0 when it is smaller than one image.
inline size_t raw_stride(uint64_t size, const Index &V) {
    const size_t tight = (size_t)V.cols * V.bpp, padded = (tight + 3) & ~(size_t)3;
    return size >= padded * V.rows ? padded : size >= tight * V.rows ? tight : 0;
}

// ---- Matroska -----------------------------------------------------------------------------------------------------------

// One EBML element header at d[0, n): the ID with its length marker, the data size without it (-1: unknown size).  Returns the
// header's length, 0 when it does not fit in n bytes, -1 when it is not a valid header.
inline int ebml_header(const uint8_t *d, size_t n, uint32_t &id, int64_t &size) {
    auto len = [](uint8_t b) {
        for (int k = 1; k <= 8; ++k)
            if (b & (0x80 >> (k - 1))) return k;
        return 0;
    };
    if (n < 1) return 0;
    const int il = len(d[0]);
    if (!il || il > 4) return -1;
    if (n < (size_t)il + 1) return 0;
    const int sl = len(d[il]);
    if (!sl) return -1;
    if (n < (size_t)(il + sl)) return 0;
    id = (uint32_t)be_n(d, (size_t)il);
    uint64_t v = d[il] & (0xFF >> sl);
    for (int k = 1; k < sl; ++k) v = (v << 8) | d[il + k];
    size = v == ((uint64_t)1 << (7 * sl)) - 1 ? -1 : (int64_t)v;
    return il + sl;
}

// The children of an element held in memory: fn(id, data, size) for each.
template <class Fail, class Fn>
void ebml_children(const uint8_t *d, size_t n, const Fail &fail, const Fn &fn) {
    for (size_t p = 0; p < n;) {
        uint32_t id;
        int64_t size;
        const int hl = ebml_header(d + p, n - p, id, size);
        if (hl <= 0 || size < 0 || (uint64_t)size > n - p - (size_t)hl) fail("truncated or invalid element inside a track or segment header");
        fn(id, d + p + hl, (size_t)size);
        p += (size_t)hl + (size_t)size;
    }
}

// av_reduce (libavutil/rational.c): the closest fraction num / den with both terms at most max.  libavformat's Matroska demuxer
// turns a track's DefaultDuration into its frame rate this way: av_reduce(1e9, DefaultDuration, 30000).
inline void reduce_rational(int64_t num, int64_t den, int64_t max, int64_t &out_num, int64_t &out_den) {
    int64_t a0n = 0, a0d = 1, a1n = 1, a1d = 0;
    int64_t a = num, b = den;
    while (b) {
        const int64_t t = a % b;
        a = b;
        b = t;
    }
    if (a) num /= a, den /= a;
    if (num <= max && den <= max) {
        a1n = num;
        a1d = den;
        den = 0;
    }
    while (den) {
        int64_t x = num / den;
        const int64_t next_den = num - den * x;
        const int64_t a2n = x * a1n + a0n, a2d = x * a1d + a0d;
        if (a2n > max || a2d > max) {
            if (a1n) x = (max - a0n) / a1n;
            if (a1d) x = std::min(x, (max - a0d) / a1d);
            if (den * (2 * x * a1d + a0d) > num * a1d) {
                a1n = x * a1n + a0n;
                a1d = x * a1d + a0d;
            }
            break;
        }
        a0n = a1n;
        a0d = a1d;
        a1n = a2n;
        a1d = a2d;
        num = den;
        den = next_den;
    }
    out_num = a1n;
    out_den = a1d;
}

}  // namespace detail

// The frame count cv::VideoCapture reports for a Matroska file (CAP_PROP_FRAME_COUNT), and so the count the reference tracks.
// Matroska stores none, so OpenCV's get_total_frames estimates floor(duration * fps + 0.5), where libavformat gives the
// duration as int64 microseconds of Duration * TimecodeScale (truncated) and the frame rate as av_reduce(1e9, DefaultDuration,
// 30000).  Pinned against cv2 in tests/test_containers.py.
inline int64_t mkv_frame_count(double duration, uint64_t timecode_scale, uint64_t default_duration) {
    const int64_t us = (int64_t)(duration * (double)timecode_scale * 1000.0 / 1000000.0);
    int64_t num, den;
    detail::reduce_rational(1000000000, (int64_t)default_duration, 30000, num, den);
    const double fps = (double)num / (double)den;
    return (int64_t)std::floor((double)us / 1000000.0 * fps + 0.5);
}

inline bool is_mkv(const std::string &name) {
    const std::vector<uint8_t> h = slurp(name, 4);
    return h.size() >= 4 && h[0] == 0x1A && h[1] == 0x45 && h[2] == 0xDF && h[3] == 0xA3;
}

inline Index index_mkv(const std::string &name, const Options &opt) {
    enum : uint32_t {
        EBML = 0x1A45DFA3, DocType = 0x4282, Segment = 0x18538067, Info = 0x1549A966, TimecodeScale = 0x2AD7B1, Duration = 0x4489,
        Tracks = 0x1654AE6B, TrackEntry = 0xAE, TrackNumber = 0xD7, TrackType = 0x83, CodecID = 0x86, CodecPrivate = 0x63A2,
        DefaultDuration = 0x23E383, Video = 0xE0, PixelWidth = 0xB0, PixelHeight = 0xBA, ColourSpace = 0x2EB524,
        ContentEncodings = 0x6D80, Cluster = 0x1F43B675, SimpleBlock = 0xA3, BlockGroup = 0xA0, Block = 0xA1
    };
    detail::File file(name);
    auto fail = [&](const std::string &why) -> void { throw std::runtime_error("Video file " + name + ": " + why); };
    const int64_t file_bytes = file.size();
    if (file_bytes < 0) fail("cannot read the file");
    struct Blk {
        uint64_t track;
        int64_t at;
        uint32_t size;
        bool laced;
    };
    struct Track {
        uint64_t number = 0, type = 0, default_duration = 0, width = 0, height = 0;
        std::string codec;
        std::vector<uint8_t> priv;
        uint8_t colour[4] = {};
        bool has_colour = false, encoded = false;
    };
    std::vector<Blk> blocks;
    std::vector<Track> tracks;
    double duration = -1;
    uint64_t timecode_scale = 1000000;
    // the entered masters (Segment, Cluster, Tracks, BlockGroup) and where each ends; one of unknown size ends with its parent
    struct Open {
        uint32_t id;
        int64_t end;
        bool unknown;
    };
    std::vector<Open> open{{0, file_bytes, false}};
    std::vector<uint8_t> buf;
    auto read_whole = [&](int64_t at, int64_t size) -> const std::vector<uint8_t> & {
        buf.resize((size_t)size);
        if (!file.seek(at) || !file.read(buf.data(), (size_t)size)) fail("truncated element at byte " + std::to_string(at));
        return buf;
    };
    for (int64_t pos = 0; pos < file_bytes;) {
        while (open.size() > 1 && pos >= open.back().end) open.pop_back();
        uint8_t h[32];
        const size_t got = (size_t)std::min<int64_t>((int64_t)sizeof h, file_bytes - pos);
        if (!file.seek(pos) || !file.read(h, got)) fail("cannot read the element at byte " + std::to_string(pos));
        uint32_t id = 0;
        int64_t size = 0;
        const int hl = detail::ebml_header(h, got, id, size);
        if (hl == 0) fail("truncated element at byte " + std::to_string(pos));
        if (hl < 0) fail("not a valid EBML element at byte " + std::to_string(pos));
        if (pos == 0 && id != EBML) fail("no EBML header");
        // a level-1 element closes a Cluster of unknown size
        if (open.back().unknown && open.back().id == Cluster && (id == Cluster || id == Info || id == Tracks || id == 0x1C53BB6B /* Cues */ ||
                                                                 id == 0x1254C367 /* Tags */ || id == 0x114D9B74 /* SeekHead */ ||
                                                                 id == 0x1043A770 /* Chapters */ || id == 0x1941A469 /* Attachments */))
            open.pop_back();
        const int64_t data = pos + hl, parent_end = open.back().end;
        if (size < 0 && id != Segment && id != Cluster) {
            char hex[16];
            std::snprintf(hex, sizeof hex, "0x%X", id);
            fail(std::string("element ") + hex + " of unknown size at byte " + std::to_string(pos) + " (only a Segment or a Cluster may have one)");
        }
        const int64_t end = size < 0 ? parent_end : data + size;
        if (end > parent_end)
            fail("truncated element at byte " + std::to_string(pos) + ": it runs past " + (open.size() == 1 ? "the end of the file" : "its parent element"));
        if (id == Segment || id == Cluster || id == Tracks || id == BlockGroup) {
            open.push_back(Open{id, end, size < 0});
            pos = data;
            continue;
        }
        if (id == EBML) {
            if (size > 4096) fail("oversized EBML header");
            std::string doctype;
            detail::ebml_children(read_whole(data, size).data(), (size_t)size, fail, [&](uint32_t cid, const uint8_t *d, size_t n) {
                if (cid == DocType) doctype.assign(reinterpret_cast<const char *>(d), strnlen(reinterpret_cast<const char *>(d), n));
            });
            if (doctype != "matroska") fail("EBML DocType '" + doctype + "': only Matroska ('matroska') files are read here");
        } else if (id == Info) {
            if (size > (1 << 20)) fail("oversized segment information");
            detail::ebml_children(read_whole(data, size).data(), (size_t)size, fail, [&](uint32_t cid, const uint8_t *d, size_t n) {
                if (cid == TimecodeScale) timecode_scale = detail::be_n(d, std::min<size_t>(n, 8));
                if (cid == Duration && n == 4) {
                    const uint32_t u = (uint32_t)detail::be_n(d, 4);
                    float f;
                    std::memcpy(&f, &u, 4);
                    duration = f;
                }
                if (cid == Duration && n == 8) {
                    const uint64_t u = detail::be_n(d, 8);
                    std::memcpy(&duration, &u, 8);
                }
            });
        } else if (id == TrackEntry) {
            if (size > (64 << 20)) fail("oversized track entry");
            Track t;
            detail::ebml_children(read_whole(data, size).data(), (size_t)size, fail, [&](uint32_t cid, const uint8_t *d, size_t n) {
                if (cid == TrackNumber) t.number = detail::be_n(d, std::min<size_t>(n, 8));
                else if (cid == TrackType) t.type = detail::be_n(d, std::min<size_t>(n, 8));
                else if (cid == CodecID) t.codec.assign(reinterpret_cast<const char *>(d), strnlen(reinterpret_cast<const char *>(d), n));
                else if (cid == CodecPrivate) t.priv.assign(d, d + n);
                else if (cid == DefaultDuration) t.default_duration = detail::be_n(d, std::min<size_t>(n, 8));
                else if (cid == ContentEncodings) t.encoded = true;
                else if (cid == Video)
                    detail::ebml_children(d, n, fail, [&](uint32_t vid, const uint8_t *v, size_t m) {
                        if (vid == PixelWidth) t.width = detail::be_n(v, std::min<size_t>(m, 8));
                        if (vid == PixelHeight) t.height = detail::be_n(v, std::min<size_t>(m, 8));
                        if (vid == ColourSpace && m == 4) std::memcpy(t.colour, v, 4), t.has_colour = true;
                    });
            });
            tracks.push_back(std::move(t));
        } else if (id == SimpleBlock || id == Block) {
            // block header: track number (an EBML size-style integer), 16-bit relative timecode, flags (bits 1-2: lacing)
            const size_t avail = got - (size_t)hl;
            int tl = 0;
            for (int k = 1; k <= 8 && avail > 0; ++k)
                if (h[hl] & (0x80 >> (k - 1))) {
                    tl = k;
                    break;
                }
            if (!tl || size < tl + 3 || avail < (size_t)tl + 3) fail("invalid block header at byte " + std::to_string(data));
            uint64_t track = h[hl] & (0xFF >> tl);
            for (int k = 1; k < tl; ++k) track = (track << 8) | h[hl + k];
            const int64_t payload = size - tl - 3;
            if (payload > 0xFFFFFFFFll) fail("oversized block at byte " + std::to_string(data));
            blocks.push_back(Blk{track, data + tl + 3, (uint32_t)payload, (h[hl + tl + 2] & 0x06) != 0});
        }
        pos = end;  // Void, CRC-32, SeekHead, Cues, Tags, Timecode, ... and the elements read above
    }
    const Track *vt = nullptr;
    for (const Track &t : tracks)
        if (t.type == 1) {
            vt = &t;
            break;
        }
    if (!vt) fail("no video track");
    if (vt->encoded) fail("the video track is compressed or encrypted (ContentEncoding), which is not read here");
    Index V;
    V.name = name;
    V.cols = (int)vt->width;
    V.rows = (int)vt->height;
    auto outside = [&](const std::string &what) {
        fail("the video track is " + what + "; only PNG, FFV1 and uncompressed 8-bit grey or 24-bit frames are read here. " + outside_this_library());
    };
    bool raw = false;
    if (vt->codec == "V_FFV1") {
        V.codec = Codec::ffv1;
        V.extradata = vt->priv;
    } else if (vt->codec == "V_MJPEG" && opt.decode_mjpeg) {
        V.codec = Codec::mjpeg;
    } else if ((vt->codec == "V_MPEG4/ISO/SP" || vt->codec == "V_MPEG4/ISO/ASP") && opt.decode_mpeg4) {
        V.codec = Codec::mpeg4;
        V.extradata = vt->priv;  // the VOL, where the writer put it there
    } else if (vt->codec == "V_MS/VFW/FOURCC") {
        // a BITMAPINFOHEADER, as in an AVI's 'strf'
        const std::vector<uint8_t> &b = vt->priv;
        if (b.size() < 40) fail("V_MS/VFW/FOURCC track whose CodecPrivate is not a BITMAPINFOHEADER");
        const int bits = b[14] | (b[15] << 8);
        const uint32_t fourcc = le32(b.data() + 16);
        const std::string fc = detail::fourcc_text(b.data() + 16);
        auto cc = [](const char *s) { return le32(reinterpret_cast<const uint8_t *>(s)); };
        if (fourcc == cc("MPNG") || fourcc == cc("png ")) {
            V.codec = Codec::png;
        } else if (fourcc == cc("FFV1")) {
            V.codec = Codec::ffv1;
            V.extradata.assign(b.begin() + 40, b.end());
        } else if (opt.decode_mjpeg && (fourcc == cc("MJPG") || fourcc == cc("mjpg"))) {
            V.codec = Codec::mjpeg;
        } else if (opt.decode_mpeg4 && mpeg4_fourcc(fourcc)) {
            V.codec = Codec::mpeg4;
            V.fourcc = fourcc;
            V.extradata.assign(b.begin() + 40, b.end());
        } else if ((fourcc == cc("Y800") || fourcc == cc("GREY") || fourcc == cc("Y8  ")) && bits == 8) {
            raw = true;
        } else if (fourcc == 0 && (bits == 24 || bits == 32)) {  // BI_RGB: BGR(A), rows top-down as libavformat reads them from Matroska (no AVI bottom-up flip)
            raw = true;
            V.grey = false;
            V.bpp = bits / 8;
        } else {
            outside("'" + fc + "' with " + std::to_string(bits) + " bits per pixel" + (mpeg4_fourcc(fourcc) ? mpeg4_opt_in() : ""));
        }
    } else if (vt->codec == "V_UNCOMPRESSED") {
        const std::string cs = vt->has_colour ? detail::fourcc_text(vt->colour) : "";
        if (cs == "Y800" || cs == "GREY" || cs == "Y8  ") {
            raw = true;
        } else if (vt->has_colour && (!std::memcmp(vt->colour, "BGR\x18", 4) || !std::memcmp(vt->colour, "RGB\x18", 4))) {
            raw = true;
            V.grey = false;
            V.bpp = 3;
            V.channel0 = vt->colour[0] == 'R' ? 2 : 0;
        } else {
            outside("uncompressed with ColourSpace '" + cs + "'");
        }
    } else {
        outside("'" + vt->codec + "'" + (vt->codec.rfind("V_MPEG4/ISO/", 0) == 0 ? mpeg4_opt_in() : ""));
    }
    if ((raw || V.codec == Codec::ffv1) && (V.rows <= 0 || V.cols <= 0)) fail("the video track has no frame size");
    for (const Blk &b : blocks) {
        if (b.track != vt->number) continue;
        const std::string frame = "frame " + std::to_string(raw ? V.raw.size() : V.coded.size());
        if (b.laced) fail(frame + ": laced blocks are not read here");
        if (raw) {
            const size_t stride = detail::raw_stride(b.size, V);
            if (!stride) fail(frame + ": block smaller than one image");
            V.raw.push_back(Index::RawChunk{b.at, b.size, stride});
        } else {
            if (b.size == 0) fail(frame + ": empty block");
            V.coded.emplace_back(b.at, b.size);
        }
    }
    V.n = (int)(raw ? V.raw.size() : V.coded.size());
    if (V.n > 0) {
        if (duration < 0 || vt->default_duration == 0)
            fail(std::string("no ") + (duration < 0 ? "segment Duration" : "DefaultDuration in the video track") +
                 ", so the frame count OpenCV would use cannot be known");
        const int64_t want = mkv_frame_count(duration, timecode_scale, vt->default_duration);
        if (want != V.n)
            fail("the video track holds " + std::to_string(V.n) + " frames, but OpenCV would count " + std::to_string(want) +
                 " from the segment's duration and the track's frame rate (frames missing, or timestamps not evenly spaced); "
                 "the reference would track a different number of frames");
    }
    finish_index(V, file);
    return V;
}

// ---- QuickTime / MP4 (ISO BMFF) -------------------------------------------------------------------------------------------

inline bool is_mov(const std::string &name) {
    const std::vector<uint8_t> h = slurp(name, 8);
    if (h.size() < 8) return false;
    for (const char *t : {"ftyp", "moov", "mdat", "wide", "free", "skip"})
        if (!std::memcmp(h.data() + 4, t, 4)) return true;
    return false;
}

namespace detail {
struct Span {
    const uint8_t *d = nullptr;
    size_t n = 0;
};
// The boxes of d[0, n): fn(type, payload); a box that runs past its parent is refused.
template <class Fail, class Fn>
void boxes(Span s, const Fail &fail, const Fn &fn) {
    for (size_t p = 0; p + 8 <= s.n;) {
        uint64_t size = be32(s.d + p);
        size_t hl = 8;
        if (size == 1) {
            if (p + 16 > s.n) fail("truncated box");
            size = be_n(s.d + p + 8, 8);
            hl = 16;
        } else if (size == 0) {
            size = s.n - p;
        }
        if (size < hl || size > s.n - p) fail("truncated '" + fourcc_text(s.d + p + 4) + "' box");
        fn(s.d + p + 4, Span{s.d + p + hl, (size_t)size - hl});
        p += (size_t)size;
    }
}
}  // namespace detail

inline Index index_mov(const std::string &name, const Options &opt) {
    using detail::Span;
    detail::File file(name);
    auto fail = [&](const std::string &why) -> void { throw std::runtime_error("Video file " + name + ": " + why); };
    const int64_t file_bytes = file.size();
    if (file_bytes < 0) fail("cannot read the file");
    std::vector<uint8_t> moov;
    bool have_moov = false;
    for (int64_t pos = 0; pos < file_bytes;) {
        uint8_t h[16];
        if (file_bytes - pos < 8 || !file.seek(pos) || !file.read(h, 8)) fail("truncated box at byte " + std::to_string(pos));
        uint64_t size = be32(h);
        int64_t hl = 8;
        if (size == 1) {
            if (file_bytes - pos < 16 || !file.read(h + 8, 8)) fail("truncated box at byte " + std::to_string(pos));
            size = detail::be_n(h + 8, 8);
            hl = 16;
        } else if (size == 0) {
            size = (uint64_t)(file_bytes - pos);
        }
        const std::string type = detail::fourcc_text(h + 4);
        if (size < (uint64_t)hl) fail("invalid size of the '" + type + "' box at byte " + std::to_string(pos));
        if (size > (uint64_t)(file_bytes - pos))
            fail("truncated '" + type + "' box at byte " + std::to_string(pos) + ": it runs past the end of the file");
        if (type == "moof") fail("fragmented MP4 ('moof' box) is not read here");
        if (type == "moov" && !have_moov) {
            if (size > ((uint64_t)1 << 31)) fail("oversized 'moov' box");
            moov.resize((size_t)size - (size_t)hl);
            if (!file.read(moov.data(), moov.size())) fail("truncated 'moov' box");
            have_moov = true;
        }
        pos += (int64_t)size;
    }
    if (!have_moov) fail("no 'moov' box");
    struct Trak {
        bool video = false;
        Span elst, stsd, stts, stsc, stsz, stco, ctts;
        bool co64 = false;
        uint32_t media_ts = 0;
    };
    uint32_t movie_ts = 0;
    Trak vt;
    bool found = false;
    auto is = [](const uint8_t *t, const char *s) { return !std::memcmp(t, s, 4); };
    detail::boxes(Span{moov.data(), moov.size()}, fail, [&](const uint8_t *t, Span b) {
        if (is(t, "mvex")) fail("fragmented MP4 ('mvex' box) is not read here");
        if (is(t, "mvhd") && b.n >= 24) movie_ts = be32(b.d + (b.d[0] == 1 ? 20 : 12));
        if (!is(t, "trak") || found) return;
        Trak k;
        std::function<void(const uint8_t *, Span)> walk = [&](const uint8_t *c, Span s) {
            if (is(c, "edts") || is(c, "mdia") || is(c, "minf") || is(c, "stbl")) {
                detail::boxes(s, fail, walk);
            } else if (is(c, "mdhd") && s.n >= 24) {
                k.media_ts = be32(s.d + (s.d[0] == 1 ? 20 : 12));
            } else if (is(c, "hdlr") && s.n >= 12 && is(s.d + 8, "vide")) {  // QuickTime's data handler ('dhlr') follows in minf
                k.video = true;
            } else if (is(c, "elst")) {
                k.elst = s;
            } else if (is(c, "stsd")) {
                k.stsd = s;
            } else if (is(c, "stts")) {
                k.stts = s;
            } else if (is(c, "stsc")) {
                k.stsc = s;
            } else if (is(c, "stsz")) {
                k.stsz = s;
            } else if (is(c, "stco") || is(c, "co64")) {
                k.stco = s;
                k.co64 = is(c, "co64");
            } else if (is(c, "ctts")) {
                k.ctts = s;
            }
        };
        detail::boxes(b, fail, walk);
        if (k.video) vt = k, found = true;
    });
    if (!found) fail("no video ('vide') track");
    // a table box: version / flags, an entry count, then `count` entries of `each` bytes
    auto table = [&](Span s, const char *what, size_t head, size_t each) -> uint32_t {
        if (!s.d) fail(std::string("the video track has no '") + what + "' box");
        if (s.n < head) fail(std::string("truncated '") + what + "' box");
        const uint32_t count = be32(s.d + head - 4);
        if ((s.n - head) / (each ? each : 1) < count) fail(std::string("truncated '") + what + "' box");
        return count;
    };
    // timing: VideoCapture applies edit lists and composition offsets, so only the identity of each is read here
    uint64_t media_dur = 0;
    {
        const uint32_t n = table(vt.stts, "stts", 8, 8);
        for (uint32_t i = 0; i < n; ++i) media_dur += (uint64_t)be32(vt.stts.d + 8 + 8 * i) * be32(vt.stts.d + 12 + 8 * i);
    }
    if (vt.ctts.d) {
        const uint32_t n = table(vt.ctts, "ctts", 8, 8);
        for (uint32_t i = 0; i < n; ++i)
            if (be32(vt.ctts.d + 12 + 8 * i)) fail("composition time offsets ('ctts') are not read here: frames would be reordered");
    }
    const uint32_t media_ts = vt.media_ts;
    if (vt.elst.d) {
        const bool v1 = vt.elst.n > 0 && vt.elst.d[0] == 1;
        const uint32_t n = table(vt.elst, "elst", 8, v1 ? 20 : 12);
        bool identity = n == 1 && movie_ts && media_ts;
        if (identity) {
            const uint8_t *e = vt.elst.d + 8;
            const uint64_t seg = v1 ? detail::be_n(e, 8) : be32(e);
            const int64_t media_time = v1 ? (int64_t)detail::be_n(e + 8, 8) : (int64_t)(int32_t)be32(e + 4);
            const uint32_t rate = be32(e + (v1 ? 16 : 8));
            // the edit covers the whole media: its duration, in whole movie ticks, is not shorter than the media's
            identity = media_time == 0 && rate == 0x10000 &&
                       (unsigned __int128)(seg + 1) * media_ts > (unsigned __int128)media_dur * movie_ts;
        }
        if (!identity) fail("an edit list other than the identity (one edit of the whole media from time 0) is not read here");
    }
    // the sample entry
    Index V;
    V.name = name;
    if (table(vt.stsd, "stsd", 8, 0) < 1 || vt.stsd.n < 8 + 86) fail("truncated 'stsd' box");
    const uint8_t *entry = vt.stsd.d + 8;
    const uint32_t entry_size = be32(entry);
    if (entry_size < 86 || entry_size > vt.stsd.n - 8) fail("truncated sample entry");
    const std::string type = detail::fourcc_text(entry + 4);
    const Span children{entry + 86, entry_size - 86};
    V.cols = (int)((entry[32] << 8) | entry[33]);
    V.rows = (int)((entry[34] << 8) | entry[35]);
    const int depth = (entry[82] << 8) | entry[83];
    auto outside = [&](const std::string &what) {
        fail("the video track is " + what + "; only PNG, FFV1 and uncompressed 8-bit grey or 24-bit frames are read here. " + outside_this_library());
    };
    bool raw = false;
    if (type == "png " || type == "MPNG") {
        V.codec = Codec::png;
    } else if (type == "jpeg" && opt.decode_mjpeg) {
        V.codec = Codec::mjpeg;
    } else if (type == "FFV1") {
        V.codec = Codec::ffv1;
        bool glbl = false;
        detail::boxes(children, fail, [&](const uint8_t *t, Span b) {
            if (is(t, "glbl") && !glbl) V.extradata.assign(b.d, b.d + b.n), glbl = true;
        });
        if (!glbl) fail("FFV1 sample entry without a 'glbl' box (the configuration record)");
    } else if (type == "raw " && depth == 40) {
        // QuickTime: depth 32 + 8 is 8-bit grey, stored inverted: libavformat reads it through a grey palette that runs from
        // white at 0 to black at 255 (and its writer stores 255 - v), so VideoCapture gives 255 - v for a stored v
        raw = true;
        V.grey = false;
        for (int i = 0; i < 256; ++i) V.palette_b[i] = (uint8_t)(255 - i);
    } else if (type == "raw " && depth == 24) {  // RGB: channel 0 of the BGR frame is the third byte
        raw = true;
        V.grey = false;
        V.bpp = 3;
        V.channel0 = 2;
    } else if (type == "mp4v") {
        // esds: ES_Descriptor (tag 3) -> DecoderConfigDescriptor (tag 4) -> objectTypeIndication; libavformat maps 0x6D to PNG
        int oti = -1;
        std::vector<uint8_t> dsi;  // DecoderSpecificInfo (tag 5): an MPEG-4 stream's VOL
        detail::boxes(children, fail, [&](const uint8_t *t, Span b) {
            if (!is(t, "esds") || b.n < 4) return;
            size_t p = 4, len = 0;
            auto descr = [&](int tag) -> bool {
                if (p >= b.n || b.d[p] != tag) return false;
                ++p;
                len = 0;
                for (int k = 0; k < 4 && p < b.n; ++k) {
                    len = (len << 7) | (b.d[p] & 0x7F);
                    if (!(b.d[p++] & 0x80)) break;
                }
                return true;
            };
            if (!descr(3) || p + 3 > b.n) return;
            const uint8_t flags = b.d[p + 2];
            p += 3;
            if (flags & 0x80) p += 2;
            if ((flags & 0x40) && p < b.n) p += 1 + b.d[p];
            if (flags & 0x20) p += 2;
            if (descr(4) && p < b.n) {
                oti = b.d[p];
                p += 13;  // objectTypeIndication, streamType, bufferSizeDB, maxBitrate, avgBitrate
                if (descr(5)) dsi.assign(b.d + p, b.d + std::min<size_t>(b.n, p + len));
            }
        });
        if (oti == 0x6C && opt.decode_mjpeg) V.codec = Codec::mjpeg;  // libavformat: 0x6C is MJPEG
        else if (oti == 0x20 && opt.decode_mpeg4) V.codec = Codec::mpeg4, V.extradata = dsi;  // 0x20: MPEG-4 Part 2 visual
        else if (oti != 0x6D) outside("'mp4v' with object type " + std::to_string(oti) + " (not PNG)" + (oti == 0x20 ? mpeg4_opt_in() : ""));
        else V.codec = Codec::png;
    } else if (type == "raw ") {
        outside("'raw ' with depth " + std::to_string(depth));
    } else {
        outside("'" + type + "'");
    }
    if ((raw || V.codec == Codec::ffv1) && (V.rows <= 0 || V.cols <= 0)) fail("the sample entry has no frame size");
    // sample offsets: chunk offsets (stco / co64), samples per chunk (stsc runs), sample sizes (stsz)
    if (!vt.stsz.d || vt.stsz.n < 12) fail("truncated 'stsz' box");
    const uint32_t one_size = be32(vt.stsz.d + 4);
    const uint32_t samples = one_size ? be32(vt.stsz.d + 8) : table(vt.stsz, "stsz", 12, 4);
    const uint32_t chunks = table(vt.stco, vt.co64 ? "co64" : "stco", 8, vt.co64 ? 8 : 4);
    const uint32_t runs = table(vt.stsc, "stsc", 8, 12);
    auto sample_size = [&](uint32_t i) { return one_size ? one_size : be32(vt.stsz.d + 12 + 4 * (size_t)i); };
    auto chunk_at = [&](uint32_t c) { return vt.co64 ? (int64_t)detail::be_n(vt.stco.d + 8 + 8 * (size_t)c, 8) : (int64_t)be32(vt.stco.d + 8 + 4 * (size_t)c); };
    std::vector<std::pair<int64_t, uint32_t>> s;
    s.reserve(samples);
    for (uint32_t r = 0; r < runs; ++r) {
        const uint8_t *e = vt.stsc.d + 8 + 12 * (size_t)r;
        const uint32_t first = be32(e), per = be32(e + 4), next = r + 1 < runs ? be32(e + 12) : chunks + 1;
        if (first < 1 || next < first || next > chunks + 1 || (r == 0 && first != 1)) fail("the 'stsc' box does not match the chunk table");
        for (uint32_t c = first; c < next; ++c) {
            int64_t at = chunk_at(c - 1);
            for (uint32_t k = 0; k < per; ++k) {
                if (s.size() >= samples) fail("the sample-to-chunk table names more samples than 'stsz' has");
                const uint32_t sz = sample_size((uint32_t)s.size());
                s.emplace_back(at, sz);
                at += sz;
            }
        }
    }
    if (s.size() != samples) fail("the sample-to-chunk table names " + std::to_string(s.size()) + " samples, 'stsz' " + std::to_string(samples));
    if (raw) {
        for (size_t i = 0; i < s.size(); ++i) {
            const size_t stride = detail::raw_stride(s[i].second, V);
            if (!stride) fail("frame " + std::to_string(i) + ": sample smaller than one image");
            V.raw.push_back(Index::RawChunk{s[i].first, s[i].second, stride});
        }
    } else {
        for (size_t i = 0; i < s.size(); ++i)
            if (s[i].second == 0) fail("frame " + std::to_string(i) + ": empty sample");
        V.coded = std::move(s);
    }
    V.n = (int)(raw ? V.raw.size() : V.coded.size());
    finish_index(V, file);
    return V;
}

}  // namespace lmmedia
