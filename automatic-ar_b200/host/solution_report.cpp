// solution_report — how good is a calibration, and where is it bad (not in the reference):
//   solution_report <in.solution> [-frames] [-q q1,q2,...] [-reject <px> <out.solution>]
// Reprojection errors of the .solution's poses against its detections (MultiCamMapper::error_report, Huber weights off): totals, exact
// percentiles of the per-detection error, one line per camera and per marker, and per frame with -frames.  -reject removes the detections
// whose error is above px (and frames left without any), solves again with the file's Config flags, writes out.solution and reports again.
// Every value is printed with %.17g; one record per line, "key value" pairs after the record name:
//   report <before|after>
//   total observations <n> not_in_problem <k> sum_sq <v> rms <px>
//   percentile <q> error <px>
//   camera|marker|frame <id> observations <n> sum_sq <v> rms <px> max <px>
#include <cstdio>
#include <iostream>
#include <sstream>
#include <string>

#include "multicam_mapper.h"

static void print_report(const char *label, const aar::MultiCamMapper::ErrorReport &r, bool frames) {
    std::printf("report %s\n", label);
    std::printf("total observations %lld not_in_problem %lld sum_sq %.17g rms %.17g\n", r.observations, r.not_in_problem, r.sum_sq,
                std::sqrt(r.sum_sq / (4.0 * (double)r.observations)));
    for (size_t i = 0; i < r.q.size(); i++) std::printf("percentile %.17g error %.17g\n", r.q[i], r.q_value[i]);
    auto lines = [](const char *what, const std::map<int, aar::MultiCamMapper::EntityError> &m) {
        for (auto &p : m)
            std::printf("%s %d observations %lld sum_sq %.17g rms %.17g max %.17g\n", what, p.first, p.second.observations, p.second.sum_sq, p.second.rms(), p.second.max);
    };
    lines("camera", r.cams);
    lines("marker", r.markers);
    if (frames) lines("frame", r.frames);
}

int main(int argc, char **argv) {
    if (argc < 2) {
        std::cout << "Usage: solution_report <in.solution> [-frames] [-q q1,q2,...] [-reject <px> <out.solution>]" << std::endl;
        return -1;
    }
    bool frames = false, reject = false; double reject_px = 0; std::string out_path;
    std::vector<double> q = {0.5, 0.9, 0.99};
    try {
        for (int i = 2; i < argc; i++) {
            const std::string a = argv[i];
            if (a == "-frames") frames = true;
            else if (a == "-q" && i + 1 < argc) {
                q.clear(); std::stringstream ss(argv[++i]); std::string t;
                while (std::getline(ss, t, ',')) if (!t.empty()) q.push_back(std::stod(t));
            } else if (a == "-reject" && i + 2 < argc) { reject = true; reject_px = std::stod(argv[++i]); out_path = argv[++i]; }
            else { std::cerr << "solution_report: unknown or incomplete option " << a << std::endl; return -1; }
        }
        aar::MultiCamMapper mcm;
        if (!mcm.read_solution_file(argv[1])) return 1;
        print_report("before", mcm.error_report(q), frames);
        if (reject) {
            aar::MultiCamMapper::Rejection rj;
            mcm.remove_outliers(reject_px, &rj);
            std::printf("removed %lld of %lld detections above %.17g px\n", rj.removed, rj.observations, reject_px);
            for (int id : rj.dropped_frames) std::printf("dropped frame %d\n", id);
            for (int id : rj.unobserved_cams) std::printf("unobserved camera %d\n", id);
            for (int id : rj.unobserved_markers) std::printf("unobserved marker %d\n", id);
            std::fflush(stdout);
            mcm.solve();
            std::cout.precision(17); std::cout << "final_error: " << mcm.final_error << " iterations: " << mcm.iterations << std::endl;
            if (!mcm.write_solution_file(out_path)) return 1;
            print_report("after", mcm.error_report(q), frames);
        }
    } catch (const std::exception &e) { std::cerr << "solution_report: " << e.what() << std::endl; return 2; }
    return 0;
}
