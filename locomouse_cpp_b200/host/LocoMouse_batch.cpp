// LocoMouse_batch.cpp — locomouse_b200_batch: the reference's main() sequence (LocoMouse_main.cpp) for every video of a
// list, in one process, on every visible GPU.
//
//   locomouse_b200_batch METHOD CONFIG LIST MODEL CALIBRATION SIDE OUTPUT_FOLDER
//
// The arguments are the reference's, with the video / background pair replaced by a list file: one video per line,
// tab-separated "video<TAB>background[<TAB>side]".  The optional side (L / R) overrides SIDE for that video; relative paths
// are resolved against the list file's directory; blank lines and lines starting with '#' are ignored.
//
// Before any CUDA call the list is checked (every file exists, every side is L or R, no two videos share an output stem, since
// they would write the same output_<stem>.yml); a refusal names the line and the program exits with EXIT_FAILURE.
//
// Every visible device (restrict with CUDA_VISIBLE_DEVICES) runs batch_workers_per_gpu workers (config key); a worker is one
// host thread owning one lm_ctx.  Videos go through one shared queue, largest file first.  While a worker runs a video, a
// reader thread reads the index and first window of its next one into the second of its two pooled page-locked buffers; a
// video longer than one window (max_resident_bytes) reads its later windows into the worker's third buffer (LocoMouse_WindowPool)
// while the device works on the one before.  So a worker holds at most three windows of frames or coded chunks in host
// memory: the host footprint is at most 3 x workers x max_resident_bytes (less for videos shorter than a window).  tracker_threads defaults to hardware threads / workers.  Each video runs exactly main()'s sequence on its worker's
// context and writes the files locomouse_b200 writes for it alone.  OUTPUT_FOLDER/batch_summary.tsv gets one row per video
// of the list: status (ok, invalid, runtime, not run), device, frames, seconds of load (file read + construction) / pass 1 /
// loop / tracks / export, and the message main() would have printed.  A failing video is recorded and the others go on; a
// runtime failure after which the device no longer answers stops that device's workers and the queue drains to the others.
// The exit code is EXIT_FAILURE when any row is not ok or the summary cannot be written.
#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <deque>
#include <fstream>
#include <future>
#include <iostream>
#include <map>
#include <memory>
#include <mutex>
#include <sstream>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "LocoMouse_class.hpp"

namespace {

using clk = std::chrono::steady_clock;
double secs(clk::time_point a, clk::time_point b) { return std::chrono::duration<double>(b - a).count(); }

struct Entry {
    int line = 0;
    std::string video, bkg, side, stem;
    int64_t bytes = 0;
    // outcome
    std::string status = "not run", message;
    int device = -1;
    unsigned int frames = 0;
    double t[5] = {0, 0, 0, 0, 0};  // load, pass 1, loop, tracks, export
};

bool regular_file(const std::string &p, int64_t *bytes = nullptr) {
    struct stat st;
    if (stat(p.c_str(), &st) != 0 || !S_ISREG(st.st_mode)) return false;
    if (bytes) *bytes = (int64_t)st.st_size;
    return true;
}

std::string trim(const std::string &s) {
    size_t a = 0, b = s.size();
    while (a < b && std::isspace((unsigned char)s[a])) ++a;
    while (b > a && std::isspace((unsigned char)s[b - 1])) --b;
    return s.substr(a, b - a);
}

// The list file's videos; every problem found is appended to `errors`, naming its line.
std::vector<Entry> read_list(const std::string &list, const std::string &cli_side, std::vector<std::string> &errors) {
    std::ifstream in(list);
    if (!in) {
        errors.push_back("Could not open the list file: " + list);
        return {};
    }
    const size_t slash = list.find_last_of('/');
    const std::string dir = slash == std::string::npos ? "" : list.substr(0, slash + 1);
    auto resolve = [&](const std::string &p) { return p.empty() || p[0] == '/' ? p : dir + p; };
    std::vector<Entry> out;
    std::map<std::string, int> stems;
    LocoMouse_ParseInputs names;
    std::string text;
    for (int line = 1; std::getline(in, text); ++line) {
        if (!text.empty() && text.back() == '\r') text.pop_back();
        const std::string t = trim(text);
        if (t.empty() || t[0] == '#') continue;
        const std::string where = "list line " + std::to_string(line) + ": ";
        std::vector<std::string> f;
        std::stringstream ss(text);
        for (std::string x; std::getline(ss, x, '\t');) f.push_back(trim(x));
        if (f.size() < 2 || f.size() > 3) {
            errors.push_back(where + "expected video<TAB>background[<TAB>side], found " + std::to_string(f.size()) + " field(s)");
            continue;
        }
        Entry e;
        e.line = line;
        e.video = resolve(f[0]);
        e.bkg = resolve(f[1]);
        e.side = f.size() == 3 ? f[2] : cli_side;
        bool ok = true;
        if (!regular_file(e.video, &e.bytes)) errors.push_back(where + "video file " + e.video + " does not exist"), ok = false;
        if (!regular_file(e.bkg)) errors.push_back(where + "background file " + e.bkg + " does not exist"), ok = false;
        if (e.side != "L" && e.side != "R")
            errors.push_back(where + "side '" + e.side + "' must be either \"L\" or \"R\"" + (f.size() == 3 ? "" : " (from the command line)")), ok = false;
        e.stem = names.stripFileName(e.video);
        const auto seen = stems.find(e.stem);
        if (seen != stems.end())
            errors.push_back(where + "output stem '" + e.stem + "' is also the stem of line " + std::to_string(seen->second) + " (both would write output_" + e.stem +
                             ".yml)"),
                ok = false;
        else
            stems[e.stem] = line;
        if (ok) out.push_back(e);
    }
    if (errors.empty() && out.empty()) errors.push_back("the list file " + list + " names no video");
    return out;
}

std::string one_line(std::string s) {
    for (char &c : s)
        if (c == '\t' || c == '\n' || c == '\r') c = ' ';
    return s;
}

bool write_summary(const std::string &folder, const std::vector<Entry> &E) {
    std::ofstream o(folder + "/batch_summary.tsv");
    o << "line\tvideo\tstatus\tdevice\tframes\tload_s\tpass1_s\tloop_s\ttracks_s\texport_s\tmessage\n";
    for (const Entry &e : E) {
        o << e.line << '\t' << one_line(e.video) << '\t' << e.status << '\t' << e.device << '\t' << e.frames;
        for (double x : e.t) o << '\t' << x;
        o << '\t' << one_line(e.message) << '\n';
    }
    o.close();
    if (o) return true;
    std::cout << "Runtime Error: could not write " << folder << "/batch_summary.tsv" << std::endl;
    return false;
}

// Videos not yet taken, largest file first; a worker whose device stopped answering puts its prefetched video back.
class Queue {
    std::mutex m_;
    std::deque<int> q_;

public:
    explicit Queue(const std::vector<Entry> &E) {
        for (size_t i = 0; i < E.size(); ++i) q_.push_back((int)i);
        std::stable_sort(q_.begin(), q_.end(), [&](int a, int b) { return E[a].bytes > E[b].bytes; });
    }
    int pop() {
        std::lock_guard<std::mutex> l(m_);
        if (q_.empty()) return -1;
        const int i = q_.front();
        q_.pop_front();
        return i;
    }
    void give_back(int i) {
        std::lock_guard<std::mutex> l(m_);
        q_.push_front(i);
    }
};

struct Shared {
    std::vector<Entry> &E;
    const LocoMouse_ParseInputs &base;  // METHOD, CONFIG, MODEL, CALIBRATION, OUTPUT and the program path
    const LocoMouse_Parameters &params;
    Queue &queue;
    std::vector<std::unique_ptr<std::atomic<bool>>> &dead;  // per device: a runtime failure left it unusable
    std::mutex &out;
};

// One worker: one host thread, one context.
void worker(Shared &S, int dev, lm_ctx *ctx) {
    LocoMouse_Media media[2];
    LocoMouse_WindowPool pool;
    struct Load {
        std::string status, message;  // empty: loaded
        double secs = 0;
    };
    auto load = [&S](int i, LocoMouse_Media *m) {
        Load r;
        const auto t0 = clk::now();
        try {
            m->load(S.E[i].video, S.E[i].bkg, (size_t)S.params.max_resident_bytes, S.params.batch_frames, S.params.decode_mjpeg != 0,
                    S.params.decode_mpeg4 != 0);
        } catch (const std::invalid_argument &e) {
            r.status = "invalid", r.message = std::string("Invalid inputs: ") + e.what();
        } catch (const std::exception &e) {
            r.status = "runtime", r.message = std::string("Runtime Error: ") + e.what();
        }
        r.secs = secs(t0, clk::now());
        return r;
    };
    int cur = S.dead[dev]->load() ? -1 : S.queue.pop();
    std::future<Load> next_load;
    if (cur >= 0) next_load = std::async(std::launch::async, load, cur, &media[0]);
    for (int slot = 0; cur >= 0; slot ^= 1) {
        Load ld = next_load.get();
        const int next = S.dead[dev]->load() ? -1 : S.queue.pop();
        if (next >= 0) next_load = std::async(std::launch::async, load, next, &media[slot ^ 1]);
        Entry &e = S.E[cur];
        e.device = dev;
        e.t[0] = ld.secs;
        bool device_failure = false;
        if (!ld.status.empty()) {
            e.status = ld.status;
            e.message = ld.message;
        } else {
            LocoMouse_ParseInputs in = S.base;
            in.VIDEO_FILE = e.video;
            in.BKG_FILE = e.bkg;
            in.FLIP_CHAR = e.side;
            in.FILE_STEM = e.stem;
            try {
                // main()'s sequence (LocoMouse_main.cpp)
                const auto t0 = clk::now();
                std::unique_ptr<LocoMouse> L = LocoMouse_Initialize(in, S.params, media[slot], ctx, &pool);
                e.frames = L->N_frames();
                const auto t1 = clk::now();
                L->getBoundingBox();
                L->initializeFeatureLoop();
                const auto t2 = clk::now();
                for (unsigned int i_frames = 0; i_frames < L->N_frames(); ++i_frames) {
                    L->readFrame();
                    L->cropBoundingBox();
                    L->detectTail();
                    L->detectBottomCandidates();
                    L->computeUnaryCostsBottom();
                    L->computePairwiseCostsBottom();
                    L->detectSideCandidates();
                    L->matchBottomSideCandidates();
                    L->storePreviousImage();
                }
                const auto t3 = clk::now();
                L->computeBottomTracks();
                L->computeSideTracks();
                const auto t4 = clk::now();
                L->exportResults();
                const auto t5 = clk::now();
                e.t[0] += secs(t0, t1);
                e.t[1] = secs(t1, t2);
                e.t[2] = secs(t2, t3);
                e.t[3] = secs(t3, t4);
                e.t[4] = secs(t4, t5);
                e.status = "ok";
            } catch (const std::invalid_argument &x) {
                e.status = "invalid", e.message = std::string("Invalid inputs: ") + x.what();
            } catch (const std::exception &x) {
                e.status = "runtime", e.message = std::string("Runtime Error: ") + x.what();
                device_failure = true;
            }
        }
        if (device_failure) {  // does the device still answer?  (a sticky CUDA error fails every later call)
            void *p = nullptr;
            if (lm_device_alloc(ctx, &p, 256) != LM_OK) S.dead[dev]->store(true);
            else lm_device_free(ctx, p);
        }
        {
            std::lock_guard<std::mutex> l(S.out);
            std::cout << "line " << e.line << " (" << e.video << ") device " << dev << ": " << e.status;
            if (!e.message.empty()) std::cout << ": " << e.message;
            std::cout << std::endl;
        }
        if (S.dead[dev]->load()) {  // nobody here runs the prefetched video: back to the queue for the other devices
            if (next >= 0) {
                next_load.get();
                S.queue.give_back(next);
            }
            break;
        }
        cur = next;
    }
    pool.release(ctx);
}

}  // namespace

int main(int argc, char *argv[]) {
    const auto t0 = clk::now();
    int return_val = EXIT_SUCCESS;
    if (argc != 8) {
        std::cout << "Invalid inputs: Invalid input list. The input should be: locomouse_b200_batch method config.yml list.tsv model_file "
                     "calibration_file side_char output_folder."
                  << std::endl;
        std::cout << "Total Elapsed time: " << secs(t0, clk::now()) << "s" << std::endl;
        return EXIT_FAILURE;
    }
    LocoMouse_ParseInputs base;
    base.LM_CALL = argv[0];
    base.METHOD = argv[1];
    base.CONFIG_FILE = argv[2];
    const std::string list = argv[3];
    base.MODEL_FILE = argv[4];
    base.CALIBRATION_FILE = argv[5];
    const std::string cli_side = argv[6];
    base.OUTPUT_PATH = argv[7];
    const size_t slash = base.LM_CALL.find_last_of("/\\");
    base.REF_PATH = slash == std::string::npos ? "./" : base.LM_CALL.substr(0, slash + 1);

    // ---- pre-flight: nothing below touches a GPU until the list, the configuration and the method are known to be good ----
    std::vector<std::string> errors;
    LocoMouse_Parameters params;
    try {
        params = LocoMouse_Parameters(base.CONFIG_FILE);
    } catch (const std::exception &e) {
        errors.push_back(e.what());
    }
    try {
        (void)std::stoi(base.METHOD);
    } catch (const std::exception &) {
        errors.push_back("method must be an integer: 0 (default), 1 (TM) or 2 (TM_DE).");
    }
    std::vector<Entry> E = read_list(list, cli_side, errors);
    if (!errors.empty()) {
        for (const std::string &m : errors) std::cout << "Invalid inputs: " << m << std::endl;
        std::cout << "Total Elapsed time: " << secs(t0, clk::now()) << "s" << std::endl;
        return EXIT_FAILURE;
    }

    // ---- one context per worker, batch_workers_per_gpu per visible device ------------------------------------------------
    std::vector<std::pair<int, lm_ctx *>> ctxs;
    std::string create_error;
    for (int dev = 0;; ++dev) {
        lm_ctx *c = nullptr;
        if (lm_create(&c, dev) != LM_OK) {  // past the last visible device (or none usable)
            if (dev == 0) create_error = lm_last_error(nullptr);
            break;
        }
        ctxs.emplace_back(dev, c);
        for (int w = 1; w < params.batch_workers_per_gpu; ++w) {
            if (lm_create(&c, dev) != LM_OK) {
                create_error = lm_last_error(nullptr);
                break;
            }
            ctxs.emplace_back(dev, c);
        }
    }
    const int n_dev = ctxs.empty() ? 0 : ctxs.back().first + 1;
    if (params.tracker_threads == 0 && !ctxs.empty())
        params.tracker_threads = (int)std::max<unsigned int>(1, std::thread::hardware_concurrency() / (unsigned int)ctxs.size());
    if (ctxs.empty()) {
        std::cout << "Runtime Error: lm_create: " << create_error << std::endl;
        for (Entry &e : E) e.message = "Runtime Error: lm_create: " + create_error;
    } else {
        Queue queue(E);
        std::vector<std::unique_ptr<std::atomic<bool>>> dead;
        for (int d = 0; d < n_dev; ++d) dead.emplace_back(new std::atomic<bool>(false));
        std::mutex out;
        Shared S{E, base, params, queue, dead, out};
        std::vector<std::thread> threads;
        for (const auto &c : ctxs) threads.emplace_back(worker, std::ref(S), c.first, c.second);
        for (std::thread &t : threads) t.join();
        for (const auto &c : ctxs) lm_destroy(c.second);
    }
    if (!write_summary(base.OUTPUT_PATH, E)) return_val = EXIT_FAILURE;  // a caller must not lose the summary unnoticed
    int ok = 0;
    double frames = 0;
    for (const Entry &e : E) {
        ok += e.status == "ok";
        frames += e.frames;
        if (e.status != "ok") return_val = EXIT_FAILURE;
    }
    const double t = secs(t0, clk::now());
    std::cout << "LM_BATCH videos=" << E.size() << " ok=" << ok << " devices=" << n_dev << " workers=" << ctxs.size() << " frames=" << frames
              << " seconds=" << t << std::endl;
    std::cout << "Total Elapsed time: " << t << "s" << std::endl;
    return return_val;
}
