// tests/facade_large_main.cpp -- the loop of nuslam/src/slam.cpp:262-319 through the C++ facade with a 100-landmark map, which the
// engine runs in large-map mode (the oracle-order kernel's shared-memory image no longer fits): predict, associateLandmark,
// initializeLandmark, update. Prints ids / state / covariance for tests/test_large_scan_gpu.py to compare with the oracle.
#include <cstdio>
#include "nuslam_b200/slam_library.hpp"

int main()
{
    using namespace slam_library;
    const int n = 100, steps = 20, meas = 7;
    colvec robot(3), map(2 * n);
    robot(0) = 0.1;
    robot(1) = -0.2;
    robot(2) = 0.3;
    mat Q(3, 3), R(2, 2);
    for (int i = 0; i < 3; ++i) Q(i, i) = 0.1;
    for (int i = 0; i < 2; ++i) R(i, i) = 0.001;
    ExtendedKalman ekf(robot, map, Q, R);
    rigid2d::Twist2D tw;
    tw.dth = 0.02;
    tw.dx = 0.007;
    for (int step = 0; step < steps; ++step)
    {
        ekf.predict(tw);
        const int seen0 = ekf.getSeenLandmarks();   // slam.cpp:251
        for (int k = 0; k < meas; ++k)
        {
            colvec z(2);
            z(0) = 1.0 + 0.25 * k;
            z(1) = -1.5 + 0.5 * k;
            int id;
            try
            {
                id = ekf.associateLandmark(z);
            }
            catch (const std::exception & e)
            {
                printf("EXC %d %d %s\n", step, k, e.what());
                continue;
            }
            printf("ID %d %d %d\n", step, k, id);
            if (id > seen0) ekf.initializeLandmark(z, id);
            else if (id < 0) continue;
            ekf.update(tw, z, id);
        }
    }
    const colvec & x = ekf.getStateVector();
    printf("X");
    for (size_t i = 0; i < x.n_elem; ++i) printf(" %.17g", x(i));
    printf("\nS");
    const mat & S = ekf.getCovariance();
    for (size_t j = 0; j < S.n_cols; ++j)
        for (size_t i = 0; i < S.n_rows; ++i) printf(" %.17g", S(i, j));
    printf("\nSEEN %d\n", ekf.getSeenLandmarks());
    return 0;
}
