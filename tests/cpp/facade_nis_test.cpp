// Exercises the NIS read-out of the C++ facade (rigid2d::EKF_SLAM::set_nis / nis / last_nis) the way a SLAM node would:
// a by-value filter copy-assigned in INIT, prediction + measurement steps, a copy that must carry the accumulators, and
// a data_association() call.  Prints "FACADE NIS OK" and exits 0 when everything holds.
#include <cmath>
#include <cstdio>
#include <vector>

#include "rigid2d/diff_drive.hpp"
#include "rigid2d/ekf_slam.hpp"

using namespace rigid2d;

#define REQUIRE(c)                                                                \
    do {                                                                          \
        if (!(c)) {                                                               \
            std::fprintf(stderr, "REQUIRE failed line %d: %s\n", __LINE__, #c);   \
            return 1;                                                             \
        }                                                                         \
    } while (0)

static void readings(EKF_SLAM& f, mat& reading, const double* lx, const double* ly, double jitter) {
    const double th = f.getStateTheta(), x = f.getStateX(), y = f.getStateY();
    for (int i = 0; i < 3; ++i) {
        const double dx = lx[i] - x + jitter * (i - 1), dy = ly[i] - y - jitter * i;
        reading(2 * i, 0) = std::cos(th) * dx + std::sin(th) * dy;
        reading(2 * i + 1, 0) = -std::sin(th) * dx + std::cos(th) * dy;
    }
}

int main() {
    EKF_SLAM slam_agent;
    slam_agent = rigid2d::EKF_SLAM(20);
    REQUIRE(slam_agent.last_status() == 0);
    slam_agent.set_nis(true);
    REQUIRE(slam_agent.last_status() == 0);
    REQUIRE(slam_agent.last_nis().empty() && slam_agent.last_status() == 0);  // no call has run with NIS on yet
    DiffDrive dd(0.16, 0.033);
    std::vector<bool> visible(20, false), known(20, false);
    for (int i = 0; i < 3; ++i) visible[i] = true;
    mat reading = zeros<mat>(40, 1);
    const double lx[3] = {0.5, 0.2, -0.3}, ly[3] = {0.1, -0.3, 0.5};
    for (int step = 0; step < 12; ++step) {
        slam_agent.prediction(dd.getBodyTwistForUpdate(10.0 * 0.025, 10.0 * 0.035));
        readings(slam_agent, reading, lx, ly, 0.002 * ((step % 3) - 1));
        slam_agent.measurement(reading, visible, known);
        REQUIRE(slam_agent.last_status() == 0);
        const std::vector<double> v = slam_agent.last_nis();
        REQUIRE(slam_agent.last_status() == 0 && v.size() == 20);
        for (int i = 0; i < 20; ++i) {
            if (step == 0 || i >= 3) {
                REQUIRE(v[i] == -1.0);  // first measurement() and invisible slots: nothing scored
            } else {
                REQUIRE(std::isfinite(v[i]) && v[i] >= 0.0);
            }
        }
    }
    std::array<double, 4> s = slam_agent.nis();
    REQUIRE(slam_agent.last_status() == 0 && s[2] == 33.0 && s[3] == 0.0 && s[0] > 0.0);

    // copy-assignment carries the NIS switch and the accumulators: both continue identically
    EKF_SLAM copy;
    copy = slam_agent;
    REQUIRE(copy.last_status() == 0);
    std::array<double, 4> c = copy.nis();
    REQUIRE(c == s);
    for (EKF_SLAM* f : {&slam_agent, &copy}) {
        f->prediction(Twist2D(0.01, Vector2D(0.02, 0.0)));
        readings(*f, reading, lx, ly, 0.003);
        f->measurement(reading, visible, known);
        REQUIRE(f->last_status() == 0);
    }
    s = slam_agent.nis();
    c = copy.nis(true);  // read, then reset
    REQUIRE(s == c && s[2] == 36.0);
    REQUIRE(copy.nis()[2] == 0.0 && slam_agent.nis()[2] == 36.0);

    // data_association(): one value per measurement
    std::vector<Vector2D> measures;
    const double x = slam_agent.getStateX(), y = slam_agent.getStateY(), th = slam_agent.getStateTheta();
    for (int i = 0; i < 3; ++i) {
        const double dx = lx[i] - x, dy = ly[i] - y;
        measures.push_back(Vector2D(std::cos(th) * dx + std::sin(th) * dy, -std::sin(th) * dx + std::cos(th) * dy));
    }
    slam_agent.data_association(measures, known);
    REQUIRE(slam_agent.last_status() == 0);
    const std::vector<double> v = slam_agent.last_nis();
    REQUIRE(v.size() == 3);
    for (double e : v) REQUIRE(e == -1.0 || std::isfinite(e));

    // switched off: the accumulators stay as they are
    slam_agent.set_nis(false);
    s = slam_agent.nis();
    slam_agent.prediction(Twist2D(0.0, Vector2D(0.01, 0.0)));
    slam_agent.measurement(reading, visible, known);
    REQUIRE(slam_agent.nis() == s);

    // a failure goes through last_status(): a default-constructed object has no filter
    EKF_SLAM empty;
    empty.set_nis(true);
    REQUIRE(empty.last_status() != 0);
    REQUIRE(empty.last_nis().empty() && empty.last_status() != 0);
    std::printf("FACADE NIS OK\n");
    return 0;
}
