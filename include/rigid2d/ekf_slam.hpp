// rigid2d::EKF_SLAM with the reference's public call surface
// (rigid2d/include/rigid2d/ekf_slam.hpp:19-57), implemented as a thin shell over the C ABI in ekf_slam_b200.h.
// The nuslam nodes (slam.cpp:213,428,433-434 / unknown_data_assoc.cpp:409-415) compile against this unchanged:
// by-value member, copy-assignment of a fresh filter in INIT, prediction / measurement / data_association,
// scalar getters and getStateLandmark().
//
// `mat` is arma::mat when <armadillo> is available (as in the reference, which also pulls namespace arma into
// the global scope), otherwise a small column-major stand-in with the accessors the callers use.
#ifndef EKF_SLAM_INCLUDE_GUARD_HPP
#define EKF_SLAM_INCLUDE_GUARD_HPP

#include <array>
#include <cstdint>
#include <cstdio>
#include <utility>
#include <vector>

#include "../ekf_slam_b200.h"
#include "rigid2d.hpp"

#if defined(__has_include)
#if __has_include(<armadillo>) && !defined(EKF_B200_NO_ARMADILLO)
#include <armadillo>
#define EKF_B200_HAVE_ARMADILLO 1
using namespace arma;
#endif
#endif

#ifndef EKF_B200_HAVE_ARMADILLO
namespace ekf_b200 {
class mat {  // column-major dense matrix of doubles: (r,c) access, n_rows / n_cols, zeros<mat>(r,c)
  public:
    unsigned long long n_rows = 0, n_cols = 0, n_elem = 0;
    mat() {}
    mat(unsigned long long r, unsigned long long c) : n_rows(r), n_cols(c), n_elem(r * c), v_(r * c, 0.0) {}
    double& operator()(unsigned long long r, unsigned long long c) { return v_[r + c * n_rows]; }
    const double& operator()(unsigned long long r, unsigned long long c) const { return v_[r + c * n_rows]; }
    double* memptr() { return v_.data(); }
    const double* memptr() const { return v_.data(); }

  private:
    std::vector<double> v_;
};
template <class M>
inline M zeros(unsigned long long r, unsigned long long c) {
    return M(r, c);
}
}  // namespace ekf_b200
using ekf_b200::mat;
using ekf_b200::zeros;
#endif

namespace rigid2d {

class EKF_SLAM {
  public:
    EKF_SLAM() {}  // empty object, like the reference's default constructor; assign a real one before use
    explicit EKF_SLAM(int n_measurements, int device = 0) { status_ = ekf_create(n_measurements, device, &h_); report("ekf_create"); }
    EKF_SLAM(const EKF_SLAM& o) { copy_from(o); }
    EKF_SLAM(EKF_SLAM&& o) noexcept : h_(o.h_), status_(o.status_) { o.h_ = nullptr; }
    EKF_SLAM& operator=(const EKF_SLAM& o) {
        if (this != &o) {
            release();
            copy_from(o);
        }
        return *this;
    }
    EKF_SLAM& operator=(EKF_SLAM&& o) noexcept {
        if (this != &o) {
            release();
            h_ = o.h_;
            status_ = o.status_;
            pose_ok_ = false;
            o.h_ = nullptr;
        }
        return *this;
    }
    ~EKF_SLAM() { release(); }

    void prediction(const rigid2d::Twist2D& twist) {
        pose_ok_ = false;
        status_ = ekf_predict(h_, twist.angular(), twist.linearX());
        report("ekf_predict");
    }

    // known_list is taken (and ignored) exactly as the reference does.
    void measurement(mat sensor_reading, std::vector<bool> visible_list, std::vector<bool> /*known_list*/) {
        const int n = ekf_num_landmarks(h_);
        if (n <= 0) return;
        std::vector<double> xy(2 * (size_t)n, 0.0);
        std::vector<uint8_t> vis((size_t)n, 0);
        for (int i = 0; i < 2 * n && i < (int)sensor_reading.n_elem; ++i) xy[i] = sensor_reading(i, 0);
        for (int i = 0; i < n && i < (int)visible_list.size(); ++i) vis[i] = visible_list[i] ? 1 : 0;
        pose_ok_ = false;
        status_ = ekf_measurement(h_, xy.data(), vis.data());
        report("ekf_measurement");
    }

    void data_association(std::vector<rigid2d::Vector2D> measures, std::vector<bool>& known_list) {
        const int n = ekf_num_landmarks(h_);
        if (n <= 0) return;
        std::vector<double> xy(2 * measures.size());
        for (size_t j = 0; j < measures.size(); ++j) {
            xy[2 * j] = measures[j].x;
            xy[2 * j + 1] = measures[j].y;
        }
        std::vector<uint8_t> known((size_t)n, 0);
        for (int i = 0; i < n && i < (int)known_list.size(); ++i) known[i] = known_list[i] ? 1 : 0;
        last_assoc_.assign(measures.size(), -1);
        pose_ok_ = false;
        status_ = ekf_data_association(h_, xy.data(), (int)measures.size(), known.data(), last_assoc_.data(), nullptr,
                                       nullptr, nullptr);
        report("ekf_data_association");
        for (int i = 0; i < n && i < (int)known_list.size(); ++i) known_list[i] = known[i] != 0;
    }

    double getStateX() { return pose(1); }
    double getStateY() { return pose(2); }
    double getStateTheta() { return pose(0); }
    mat getStateLandmark() {
        const int n = ekf_num_landmarks(h_);
        mat out = zeros<mat>(n > 0 ? 2 * n : 0, 1);
        if (n > 0) {
            status_ = ekf_get_landmarks(h_, out.memptr());
            report("ekf_get_landmarks");
        }
        return out;
    }

    // not in the reference: last C-ABI status (0 = ok) and the association log of the last data_association()
    int last_status() const { return status_; }
    const std::vector<int32_t>& last_association() const { return last_assoc_; }
    // not in the reference: CSV log of every association decision (ekf_slam_b200.h); nullptr closes it
    void set_association_log(const char* path) {
        status_ = ekf_association_log_open(h_, path);
        report("ekf_association_log_open");
    }
    // not in the reference: process noise q = {theta, x, y} and measurement noise r = {range, bearing} variances
    // (ekf_set_noise); both nullptr restore the reference's values, one nullptr keeps that part at them
    void set_noise(const double q[3], const double r[2]) {
        if (!q && !r) {
            status_ = ekf_set_noise(h_, nullptr);
        } else {
            const double row[5] = {q ? q[0] : EKF_DEFAULT_Q, q ? q[1] : EKF_DEFAULT_Q, q ? q[2] : EKF_DEFAULT_Q,
                                   r ? r[0] : EKF_DEFAULT_R, r ? r[1] : EKF_DEFAULT_R};
            status_ = ekf_set_noise(h_, row);
        }
        report("ekf_set_noise");
    }
    // not in the reference: normalised innovation squared of the following measurement() / data_association() calls
    // (ekf_set_nis); copies of this object carry the switch and the accumulators
    void set_nis(bool on) {
        status_ = ekf_set_nis(h_, on ? 1 : 0);
        report("ekf_set_nis");
    }
    // {sum NIS, sum NIS^2, #scored, #non-finite} (ekf_nis); reset zeroes them after the read.  Zeros on failure.
    std::array<double, 4> nis(bool reset = false) {
        std::array<double, 4> out = {0.0, 0.0, 0.0, 0.0};
        status_ = ekf_nis(h_, out.data(), reset ? 1 : 0);
        report("ekf_nis");
        if (status_ != 0) out = {0.0, 0.0, 0.0, 0.0};
        return out;
    }
    // NIS per slot (after measurement()) or per measurement (after data_association()) of the last call that ran with
    // NIS on, -1 where nothing was scored (ekf_last_nis).  Empty on failure.
    std::vector<double> last_nis() {
        int count = 0;
        status_ = ekf_last_nis(h_, nullptr, &count);
        std::vector<double> out(status_ == 0 ? (size_t)count : 0);
        if (status_ == 0 && count > 0) status_ = ekf_last_nis(h_, out.data(), &count);
        report("ekf_last_nis");
        if (status_ != 0) out.clear();
        return out;
    }
    ekf_filter* handle() {
        pose_ok_ = false;  // the caller may change the filter behind this object
        return h_;
    }

  private:
    ekf_filter* h_ = nullptr;
    int status_ = 0;
    std::vector<int32_t> last_assoc_;

    // The nodes read x, y and theta one after the other (slam.cpp:433-434): one device read serves all three.
    double pose_[3] = {0.0, 0.0, 0.0};
    bool pose_ok_ = false;
    double pose(int k) {
        if (!pose_ok_) {
            pose_[0] = pose_[1] = pose_[2] = 0.0;
            status_ = ekf_get_pose(h_, pose_);
            report("ekf_get_pose");
            pose_ok_ = status_ == 0;
        }
        return pose_[k];
    }
    void copy_from(const EKF_SLAM& o) {
        h_ = nullptr;
        pose_ok_ = false;
        status_ = o.h_ ? ekf_clone(o.h_, &h_) : 0;
        report("ekf_clone");
    }
    void release() {
        if (h_) ekf_destroy(h_);
        h_ = nullptr;
    }
    // The reference has no error channel at all (no return codes, no exceptions); failures are logged, never thrown.
    void report(const char* what) const {
        if (status_ != 0) std::fprintf(stderr, "[ekf_slam_b200] %s failed (%d): %s\n", what, status_, ekf_last_error());
    }
};

}  // namespace rigid2d
#endif
