// Prints what the host design module (jaero_b200/csrc/host_design.cpp) computes, for tests/test_host_design_cpu.py:
//   rrc | trig | scrambler | plan <mode of PLAN_MODES> | pchannel <fb> | rt <fb>
#include "../../jaero_b200/csrc/host_design.h"
#include "plan_dump.h"
#include <cstdlib>
#include <cstring>
#include <string>

using namespace jb;

static int fail(const char *msg) { fprintf(stderr, "%s\n", msg); return 1; }

int main(int argc, char **argv)
{
    const std::string what = argc > 1 ? argv[1] : "";
    if (what == "rrc") {
        std::vector<double> t = rrc_taps(1.0, 55, 48000, 5250);
        dump_v("rrc", t.data(), t.size());
    } else if (what == "trig") {
        std::vector<double> sn, cs;
        trig_tables(sn, cs);
        dump_v("sin", sn.data(), sn.size()); dump_v("cos", cs.data(), cs.size());
    } else if (what == "scrambler") {
        for (uint8_t b : scrambler_sequence(5000)) printf("%d\n", b);
    } else if (what == "plan" && argc > 2) {
        for (const PlanMode &m : PLAN_MODES) {
            if (strcmp(m.name, argv[2])) continue;
            jaero_settings s = {m.kind, m.fft_power, m.fc, m.lockingbw, m.fb, m.Fs, m.thr, 0, 0, 0, 1};
            if (!m.burst) {
                BatchPlan b;
                if (const char *e = batch_plan(&s, 5, b)) return fail(e);
                auto c = [](const cvec &v) { return v.empty() ? nullptr : reinterpret_cast<const double2 *>(v.data()); };
                dump_batch(b.p, b.cfe, b.st_freq, c(b.cfe_tw), b.cfe_window.empty() ? nullptr : b.cfe_window.data(), c(b.pre_H), c(b.pre_tw));
            } else {
                BurstPlan b;
                if (const char *e = burst_plan(&s, 5, m.kind, b)) return fail(e);
                auto c = [](const cvec &v) { return reinterpret_cast<const double2 *>(v.data()); };
                dump_burst(b.p, b.hil, b.freq_center, b.w_btd1.data(), b.w_btdiff.data(), b.w_a1.data(), c(b.hil_H), c(b.hil_tw), c(b.tw32k));
            }
            return 0;
        }
        return fail("unknown mode");
    } else if (what == "pchannel" && argc > 2) {
        PChanParams pp;
        if (const char *e = pchannel_plan(5, atof(argv[2]), pp)) return fail(e);
        dump_pchannel(pp);
    } else if (what == "rt" && argc > 2) {
        RtParams rp;
        if (const char *e = rt_plan(atof(argv[2]), 5, rp)) return fail(e);
        dump_rt(rp);
    } else {
        return fail("usage: host_design_driver rrc | trig | scrambler | plan <mode> | pchannel <fb> | rt <fb>");
    }
    return 0;
}
