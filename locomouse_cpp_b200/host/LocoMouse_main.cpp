// LocoMouse_main.cpp — the reference's driver (main.cpp:36-106) against the B200 class mirror: same
// argument list, same call sequence, same exception handling and exit codes.
#include <chrono>
#include <cstdlib>
#include <iostream>
#include <memory>
#include <stdexcept>

#include "LocoMouse_class.hpp"

int main(int argc, char *argv[]) {
    const auto t0 = std::chrono::steady_clock::now();
    int return_val = EXIT_SUCCESS;
    using clk = std::chrono::steady_clock;
    auto secs = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double>(b - a).count(); };
    try {
        LocoMouse_ParseInputs inputs = LocoMouse_ParseInputs(argc, argv);
        std::unique_ptr<LocoMouse> L = LocoMouse_Initialize(inputs);
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
        auto t3 = clk::now();
        // LM_DRIVER_REPEAT=k: run the per-frame loop k more times on the same object (initializeFeatureLoop() rewinds the video, as
        // in the reference) and report the last one: the loop of a warm process, without CUDA module load and scratch allocation
        double warm_loop_s = -1.0;
        if (const char *e = std::getenv("LM_DRIVER_REPEAT")) {
            for (int rep = 0; rep < std::atoi(e); ++rep) {
                L->initializeFeatureLoop();
                const auto w0 = clk::now();
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
                warm_loop_s = secs(w0, clk::now());
            }
            t3 = clk::now();
        }
        L->computeBottomTracks();
        L->computeSideTracks();
        const auto t4 = clk::now();
        L->exportResults();
        const auto t5 = clk::now();
        // phases of the reference's main(): construction (file loading), pass 1, the per-frame loop, the tracker, export
        // windows: how many pieces the video was read, decoded and tracked in (max_resident_bytes); resident_bytes: the page-locked
        // bytes of frames held at the peak plus the device bytes of decoded frames; guard_violations: -1 unless LM_GUARD=1
        double guard = -1;
        lm_get_info(L->context(), "guard_violations", &guard);
        std::cout << "LM_TIMING frames=" << L->N_frames() << " load_s=" << secs(t0, t1) << " pass1_s=" << secs(t1, t2) << " loop_s=" << secs(t2, t3)
                  << " tracks_s=" << secs(t3, t4) << " export_s=" << secs(t4, t5) << " warm_loop_s=" << warm_loop_s << " windows=" << L->windows()
                  << " resident_bytes=" << L->residentBytes() << " guard_violations=" << guard << std::endl;
    } catch (const std::invalid_argument &e) {
        std::cout << "Invalid inputs: " << e.what() << std::endl;
        return_val = EXIT_FAILURE;
    } catch (const std::runtime_error &e) {
        std::cout << "Runtime Error: " << e.what() << std::endl;
        return_val = EXIT_FAILURE;
    }
    const double t = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    std::cout << "Total Elapsed time: " << t << "s" << std::endl;
    return return_val;
}
