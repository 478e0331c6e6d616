// test_host_api.cpp -- the reference's own gtest cases for the linear path
// (mav_trajectory_generation/test/test_polynomial_optimization.cpp), re-stated against the
// B200-backed PolynomialOptimization<N>.  `--cpu-only` runs the cases that need no device
// (value types, fixtures, static helpers, layout); without it every solve goes through the GPU.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <sstream>
#include <fstream>
#include <random>
#include <string>
#include <vector>

#include <unistd.h>

#include "mav_trajectory_generation/batch_polynomial_optimization.h"
#include "mav_trajectory_generation/io.h"
#include "mav_trajectory_generation/polynomial_optimization_linear.h"
#include "mav_trajectory_generation/trajectory_sampling.h"
#include "mav_trajectory_generation_ros/ros_conversions.h"

using namespace mav_trajectory_generation;

static int g_failures = 0, g_checks = 0;
#define EXPECT(cond)                                                        \
  do {                                                                      \
    ++g_checks;                                                             \
    if (!(cond)) {                                                          \
      ++g_failures;                                                         \
      std::printf("EXPECT failed %s:%d: %s\n", __FILE__, __LINE__, #cond);  \
    }                                                                       \
  } while (0)
#define EXPECT_NEAR(a, b, tol)                                                                     \
  do {                                                                                             \
    ++g_checks;                                                                                    \
    if (!(std::abs((a) - (b)) <= (tol))) {                                                         \
      ++g_failures;                                                                                \
      std::printf("EXPECT_NEAR failed %s:%d: %.17g vs %.17g (tol %g)\n", __FILE__, __LINE__,       \
                  double(a), double(b), double(tol));                                              \
    }                                                                                              \
  } while (0)

constexpr int N = 10;

struct Params {
  int D, max_derivative, num_segments, seed;
  double pos_bounds, v_max, a_max;
};
// test_polynomial_optimization.cpp:790-867
static const Params kParams[] = {
    {1, 4, 1, 100, 10.0, 3.0, 5.0},  {1, 4, 10, 102, 10.0, 3.0, 5.0}, {1, 4, 50, 103, 10.0, 3.0, 5.0},
    {3, 4, 1, 104, 10.0, 3.0, 5.0},  {3, 4, 10, 105, 10.0, 3.0, 5.0}, {3, 4, 50, 106, 10.0, 3.0, 5.0},
    {1, 2, 5, 107, 10.0, 1.0, 2.0},  {3, 2, 1, 108, 10.0, 1.0, 2.0},  {3, 2, 5, 109, 10.0, 1.0, 2.0},
    {3, 3, 5, 110, 10.0, 1.0, 2.0},
};

static Vertex::Vector fixtureVertices(const Params& p) {
  Eigen::VectorXd lo = Eigen::VectorXd::Constant(p.D, -p.pos_bounds), hi = Eigen::VectorXd::Constant(p.D, p.pos_bounds);
  return createRandomVertices(getHighestDerivativeFromN(N), p.num_segments, lo, hi, p.seed);
}

// checkPath (test :113-174)
static void checkPath(const Vertex::Vector& vertices, const std::vector<Segment>& segments) {
  const double tol = 1e-6;
  EXPECT(segments.size() == vertices.size() - 1);
  for (size_t i = 0; i < segments.size(); ++i) {
    const Segment& segment = segments[i];
    for (int end = 0; end < 2; ++end) {
      const Vertex& v = vertices[i + end];
      const double t = end ? segment.getTime() : 0.0;
      for (auto it = v.cBegin(); it != v.cEnd(); ++it) {
        const Eigen::VectorXd actual = segment.evaluate(t, it->first);
        for (int d = 0; d < segment.D(); ++d) EXPECT_NEAR(it->second[d], actual[d], tol);
      }
    }
    if (i > 0)
      for (int derivative = 0; derivative < N / 2; ++derivative) {
        const Eigen::VectorXd a = segments[i - 1].evaluate(segments[i - 1].getTime(), derivative);
        const Eigen::VectorXd b = segment.evaluate(0, derivative);
        for (int d = 0; d < segment.D(); ++d) EXPECT_NEAR(a[d], b[d], tol);
      }
  }
}

static double costNumeric(const Trajectory& trajectory, int derivative, double dt) {
  double cost = 0.0;
  for (const Segment& s : trajectory.segments())
    for (double t = 0.0; t < s.getTime(); t += dt) cost += s.evaluate(t, derivative).squaredNorm() * dt;
  return cost;
}

static void testValueTypesAndFixtures() {
  // createRandomVertices with std::mt19937(105): first vertex (SURVEY.md appendix B.8)
  Vertex::Vector v = fixtureVertices(kParams[4]);
  Eigen::VectorXd p0;
  EXPECT(v.size() == 11);
  EXPECT(v[0].getConstraint(derivative_order::POSITION, &p0));
  EXPECT(p0[0] == -3.4346932681103235 && p0[1] == 7.0047000485169981 && p0[2] == 2.9909075836621035);
  EXPECT(v[0].getNumberOfConstraints() == 5 && v[5].getNumberOfConstraints() == 1 && v[10].hasConstraint(4));
  // README example times (v = a = 2)
  Vertex::Vector r;
  Vertex s(3), m(3), e(3);
  s.makeStartOrEnd(Eigen::Vector3d(0, 0, 1), derivative_order::SNAP);
  m.addConstraint(derivative_order::POSITION, Eigen::Vector3d(1, 2, 3));
  e.makeStartOrEnd(Eigen::Vector3d(2, 1, 5), derivative_order::SNAP);
  r = {s, m, e};
  const std::vector<double> t = estimateSegmentTimes(r, 2.0, 2.0);
  EXPECT_NEAR(t[0], 3.97084783, 5e-9);
  EXPECT_NEAR(t[1], 3.82413014, 5e-9);
  // Polynomial: derivative coefficients and Horner evaluation
  Eigen::VectorXd c(4);
  c[0] = 1; c[1] = 2; c[2] = 3; c[3] = 4;
  Polynomial poly(4, c);
  EXPECT_NEAR(poly.evaluate(2.0, 0), 1 + 4 + 12 + 32, 1e-12);
  EXPECT_NEAR(poly.evaluate(2.0, 1), 2 + 12 + 48, 1e-12);
  EXPECT_NEAR(poly.getCoefficients(2)[1], 24.0, 0);
  EXPECT(Polynomial::base_coefficients_(3, 5) == 60.0);
  Eigen::VectorXd conv = Polynomial::convolve(c, c);
  EXPECT(conv.size() == 7 && conv[6] == 16.0 && conv[0] == 1.0);
}

// YAML schema of the reference (src/io.cpp:126-219): round trip and a hand-written file in the reference layout.
static void testYamlIo() {
  Segment::Vector segments;
  for (int i = 0; i < 3; ++i) {
    Segment s(10, 3);
    s.setTimeNSec(3970847830ull + 17ull * i);
    for (int d = 0; d < 3; ++d) {
      Eigen::VectorXd c(10);
      for (int j = 0; j < 10; ++j) c[j] = std::sin(1.0 + i * 31 + d * 7 + j) * std::pow(10.0, -j);
      s[d] = Polynomial(10, c);
    }
    segments.push_back(s);
  }
  const std::string yaml = segmentsToYamlString(segments);
  Segment::Vector back;
  EXPECT(segmentsFromYamlString(yaml, &back));
  EXPECT(back.size() == segments.size());
  for (size_t i = 0; i < back.size() && i < segments.size(); ++i) {
    EXPECT(back[i].getTimeNSec() == segments[i].getTimeNSec());
    for (int d = 0; d < 3; ++d) EXPECT(back[i][d] == segments[i][d]);  // %.17g round-trips bit-exactly
  }
  const std::string reference_style =
      "segments:\n"
      "  - N: 4\n"
      "    D: 2\n"
      "    time: 1500000000  # [ns]\n"
      "    coefficients:\n"
      "      - [0, 1, 0.5, -0.25]\n"
      "      - [2, 0, 0, 1e-3]\n";
  EXPECT(segmentsFromYamlString(reference_style, &back));
  EXPECT(back.size() == 1 && back[0].N() == 4 && back[0].D() == 2);
  EXPECT_NEAR(back[0].getTime(), 1.5, 1e-12);
  EXPECT_NEAR(back[0][1].getCoefficients()[3], 1e-3, 0);
  EXPECT(!segmentsFromYamlString("trajectory:\n  - N: 4\n", &back));              // no segments element
  EXPECT(!segmentsFromYamlString("segments:\n  - N: 4\n    D: 2\n", &back));       // missing elements
  EXPECT(!segmentsFromYamlString(
      "segments:\n  - N: 4\n    D: 1\n    time: 5\n    coefficients:\n      - [1, 2, 3]\n", &back));  // N mismatch
}

// AMatrixInversion (test :731-741) -- here A^-1 comes from the exact table scaling.
static void testAMatrixInversion() {
  for (double t = 1; t <= 60; t += 1) {
    PolynomialOptimization<N>::SquareMatrix A, Ai;
    PolynomialOptimization<N>::setupMappingMatrix(t, &A);
    PolynomialOptimization<N>::invertMappingMatrix(A, &Ai);
    // A * Ai == I, scaled per column of A (entries span 18 orders of magnitude at t = 60)
    for (int i = 0; i < N; ++i)
      for (int j = 0; j < N; ++j) {
        double s = 0.0, mag = 0.0;
        for (int k = 0; k < N; ++k) {
          s += A(i, k) * Ai(k, j);
          mag += std::abs(A(i, k) * Ai(k, j));
        }
        EXPECT_NEAR(s, i == j ? 1.0 : 0.0, 1e-12 * (1.0 + mag));
      }
  }
  PolynomialOptimization<N>::SquareMatrix Q;
  PolynomialOptimization<N>::computeQuadraticCostJacobian(4, 2.0, &Q);
  EXPECT(Q(3, 3) == 0.0);
  EXPECT_NEAR(Q(4, 4), 2.0 * 24 * 24 * 2.0, 1e-9);  // 2 * B(4,4)^2 * T^1 / 1
}

// Extrema machinery (reference test_polynomial.cpp / test_polynomial_optimization.cpp extrema cases restated):
// roots of a polynomial with known roots, min/max against dense sampling, magnitude extrema of a random
// multi-dimensional segment, time scaling to meet v/a limits, message round trip, evaluateRange conventions.
static void testExtremaAndConversions() {
  // p(t) = (t-1)(t-2.5)(t^2+1)(t+3) = expand: roots 1, 2.5, -3, +-i
  {
    // (t-1)(t-2.5) = t^2 - 3.5 t + 2.5 ; times (t+3) = t^3 - 0.5 t^2 - 8 t + 7.5 ; times (t^2+1)
    // = t^5 - 0.5 t^4 - 7 t^3 + 7 t^2 - 8 t + 7.5
    Eigen::VectorXd c(6);
    c[0] = 7.5; c[1] = -8.0; c[2] = 7.0; c[3] = -7.0; c[4] = -0.5; c[5] = 1.0;
    Polynomial p(6, c);
    Eigen::VectorXcd roots;
    EXPECT(p.getRoots(0, &roots));
    EXPECT(roots.size() == 5);
    int n_real = 0;
    bool got1 = false, got25 = false, gotm3 = false;
    for (Eigen::Index i = 0; i < roots.size(); ++i) {
      if (roots[i].imag() == 0.0) {
        ++n_real;
        got1 |= std::abs(roots[i].real() - 1.0) < 1e-12;
        got25 |= std::abs(roots[i].real() - 2.5) < 1e-12;
        gotm3 |= std::abs(roots[i].real() + 3.0) < 1e-12;
      } else {
        EXPECT_NEAR(std::abs(roots[i].imag()), 1.0, 1e-12);
        EXPECT_NEAR(roots[i].real(), 0.0, 1e-12);
      }
    }
    EXPECT(n_real == 3 && got1 && got25 && gotm3);
    // min / max of p on [0, 3] against dense sampling
    std::pair<double, double> lo, hi;
    EXPECT(p.computeMinMax(0.0, 3.0, 0, &lo, &hi));
    double s_lo = 1e300, s_hi = -1e300;
    for (int k = 0; k <= 300000; ++k) {
      const double v = p.evaluate(3.0 * k / 300000.0, 0);
      s_lo = std::min(s_lo, v);
      s_hi = std::max(s_hi, v);
    }
    EXPECT_NEAR(lo.second, s_lo, 1e-8);
    EXPECT_NEAR(hi.second, s_hi, 1e-8);
    EXPECT(lo.second <= s_lo + 1e-12 && hi.second >= s_hi - 1e-12);
  }
  // random 3-D segments: analytic magnitude extrema of velocity / acceleration bound the sampled ones
  std::mt19937 rng(7);
  std::uniform_real_distribution<double> u(-1.0, 1.0);
  Segment::Vector segs;
  for (int trial = 0; trial < 5; ++trial) {
    Segment seg(N, 3);
    for (int d = 0; d < 3; ++d) {
      Eigen::VectorXd c(N);
      double scale = 1.0;
      for (int j = 0; j < N; ++j) {
        c[j] = u(rng) * scale;
        scale *= 0.5;
      }
      seg[d].setCoefficients(c);
    }
    seg.setTime(2.0 + trial);
    segs.push_back(seg);
    for (int der = 1; der <= 2; ++der) {
      std::vector<double> times;
      EXPECT(PolynomialOptimization<N>::computeSegmentMaximumMagnitudeCandidates(der, seg, 0.0, seg.getTime(), &times));
      double best = 0.0;
      for (double t : times) best = std::max(best, seg.evaluate(t, der).norm());
      double sampled = 0.0;
      for (int k = 0; k <= 20000; ++k) sampled = std::max(sampled, seg.evaluate(seg.getTime() * k / 20000.0, der).norm());
      EXPECT(best >= sampled - 1e-9);
      EXPECT_NEAR(best, sampled, 1e-6 * (1.0 + sampled));
    }
  }
  Trajectory traj;
  traj.setSegments(segs);
  double v_max = 0.0, a_max = 0.0;
  EXPECT(traj.computeMaxVelocityAndAcceleration(&v_max, &a_max));
  EXPECT(v_max > 0.0 && a_max > 0.0);
  Trajectory scaled = traj;
  EXPECT(scaled.scaleSegmentTimesToMeetConstraints(0.5 * v_max, 0.25 * a_max));
  double v2 = 0.0, a2 = 0.0;
  EXPECT(scaled.computeMaxVelocityAndAcceleration(&v2, &a2));
  EXPECT(v2 <= 0.5 * v_max * 1.001 + 1e-12 && a2 <= 0.25 * a_max * 1.001 + 1e-12);
  EXPECT(scaled.getMaxTime() > traj.getMaxTime());
  // the path itself is unchanged by time scaling: same position at the same fraction of every segment
  {
    const double f = scaled.getMaxTime() / traj.getMaxTime();
    for (int k = 0; k <= 10; ++k) {
      const double t = traj.getMaxTime() * k / 10.0 * 0.999;
      const Eigen::VectorXd a = traj.evaluate(t, 0), b = scaled.evaluate(t * f, 0);
      for (int d = 0; d < 3; ++d) EXPECT_NEAR(a[d], b[d], 1e-9);
    }
  }
  // message round trip (3-D and 4-D); 5-D is rejected
  {
    mav_planning_msgs::PolynomialTrajectory msg;
    EXPECT(trajectoryToPolynomialTrajectoryMsg(traj, &msg));
    EXPECT(msg.segments.size() == segs.size() && msg.segments[0].num_coeffs == N && msg.segments[0].yaw.empty());
    EXPECT(msg.segments[1].segment_time_ns == segs[1].getTimeNSec());
    Trajectory back;
    EXPECT(polynomialTrajectoryMsgToTrajectory(msg, &back));
    EXPECT(back == traj);
    Segment s4(N, 4), s5(N, 5);
    s4.setTime(1.5);
    s5.setTime(1.5);
    Trajectory t4, t5;
    t4.setSegments(Segment::Vector(1, s4));
    t5.setSegments(Segment::Vector(1, s5));
    mav_planning_msgs::PolynomialTrajectory4D m4;
    EXPECT(trajectoryToPolynomialTrajectoryMsg(t4, &m4) && m4.segments[0].yaw.size() == size_t(N));
    Trajectory b4;
    EXPECT(polynomialTrajectoryMsgToTrajectory(m4, &b4) && b4.D() == 4);
    EXPECT(!trajectoryToPolynomialTrajectoryMsg(t5, &msg) && msg.segments.empty());
  }
  // evaluateRange follows the reference's walk: t_end is excluded, the clock starts at the start of the segment
  // that contains t_start, a start beyond the end yields nothing
  {
    std::vector<Eigen::VectorXd> out;
    std::vector<double> st;
    traj.evaluateRange(0.0, 1.0, 0.25, 0, &out, &st);
    EXPECT(out.size() == 4 && st.size() == 4 && st[3] == 0.75);
    traj.evaluateRange(traj.getMaxTime() + 1.0, traj.getMaxTime() + 2.0, 0.1, 0, &out, &st);
    EXPECT(out.empty());
    const double t0 = segs[0].getTime() + 0.5;  // inside segment 1: the sample clock starts at segs[0].getTime()
    traj.evaluateRange(t0, t0 + 1.0, 0.5, 0, &out, &st);
    EXPECT(!st.empty() && st[0] == segs[0].getTime());
    const Eigen::VectorXd direct = traj.evaluate(t0, 0);
    for (int d = 0; d < 3; ++d) EXPECT_NEAR(out[0][d], direct[d], 1e-12);
  }
  // invertMappingMatrix inverts the matrix it is given (a mapping matrix with a perturbed lower block)
  {
    PolynomialOptimization<N>::SquareMatrix A, Ai;
    PolynomialOptimization<N>::setupMappingMatrix(2.0, &A);
    for (int i = N / 2; i < N; ++i)
      for (int j = 0; j < N; ++j) A(i, j) *= 1.0 + 0.01 * ((i * 7 + j * 3) % 5);
    PolynomialOptimization<N>::invertMappingMatrix(A, &Ai);
    for (int i = 0; i < N; ++i)
      for (int j = 0; j < N; ++j) {
        double s = 0.0, mag = 0.0;
        for (int k = 0; k < N; ++k) {
          s += A(i, k) * Ai(k, j);
          mag += std::abs(A(i, k) * Ai(k, j));
        }
        EXPECT_NEAR(s, i == j ? 1.0 : 0.0, 1e-11 * (1.0 + mag));
      }
  }
}

// Trajectory re-shaping and vertex extraction (reference trajectory.h:86-124): pure host code, no GPU.
static Trajectory randomTrajectory(int K, int D, int N, unsigned seed, const std::vector<double>& times) {
  std::mt19937 gen(seed);
  std::uniform_real_distribution<double> coef(-1.0, 1.0);
  Segment::Vector segs;
  for (int k = 0; k < K; ++k) {
    Segment sgm(N, D);
    for (int d = 0; d < D; ++d) {
      Eigen::VectorXd c(N);
      for (int j = 0; j < N; ++j) c[j] = coef(gen);
      sgm[d] = Polynomial(N, c);
    }
    sgm.setTime(times[k]);
    segs.push_back(sgm);
  }
  Trajectory t;
  t.setSegments(segs);
  return t;
}

static void testTrajectoryReshaping() {
  const std::vector<double> times = {1.5, 0.75, 2.25};
  const Trajectory full = randomTrajectory(3, 4, 6, 11, times);
  const double probe[] = {0.0, 0.4, 1.5, 1.9, 2.25, 3.0, 4.5};
  // single dimension keeps the segment times and the polynomial
  for (int d = 0; d < 4; ++d) {
    const Trajectory one = full.getTrajectoryWithSingleDimension(d);
    EXPECT(one.D() == 1 && one.N() == 6 && one.K() == 3);
    EXPECT_NEAR(one.getMaxTime(), full.getMaxTime(), 0.0);
    for (double t : probe)
      for (int der = 0; der < 3; ++der) EXPECT_NEAR(one.evaluate(t, der)[0], full.evaluate(t, der)[d], 0.0);
  }
  // position (dimensions 0..2) + yaw (dimension 3) re-assembled dimension by dimension equals the original
  {
    Trajectory acc;
    for (int d = 0; d < 4; ++d) {
      Trajectory next;
      EXPECT(acc.getTrajectoryWithAppendedDimension(full.getTrajectoryWithSingleDimension(d), &next));
      acc = next;
    }
    EXPECT(acc == full);
    Trajectory same;
    EXPECT(full.getTrajectoryWithAppendedDimension(Trajectory(), &same));
    EXPECT(same == full);
    // different polynomial orders: the result carries the larger one and still evaluates to both parts
    const Trajectory low = randomTrajectory(3, 1, 4, 12, times);
    Trajectory mixed;
    EXPECT(full.getTrajectoryWithAppendedDimension(low, &mixed));
    EXPECT(mixed.D() == 5 && mixed.N() == 6);
    for (double t : probe) {
      EXPECT_NEAR(mixed.evaluate(t, 1)[4], low.evaluate(t, 1)[0], 1e-15);
      EXPECT_NEAR(mixed.evaluate(t, 0)[2], full.evaluate(t, 0)[2], 0.0);
    }
    // a shorter-lived segment of the appended trajectory is stretched to the longer duration (src/segment.cpp:218-231)
    const Trajectory other_times = randomTrajectory(3, 1, 6, 13, {1.5, 0.5, 2.25});
    Trajectory stretched;
    EXPECT(full.getTrajectoryWithAppendedDimension(other_times, &stretched));
    EXPECT_NEAR(stretched.getMaxTime(), full.getMaxTime(), 0.0);
    EXPECT_NEAR(stretched.evaluate(1.5 + 0.75 * 0.4, 0)[4], other_times.evaluate(1.5 + 0.5 * 0.4, 0)[0], 1e-14);
    EXPECT_NEAR(stretched.evaluate(1.5 + 0.75 * 0.4, 0)[1], full.evaluate(1.5 + 0.75 * 0.4, 0)[1], 0.0);
  }
  // concatenation in time
  {
    const Trajectory second = randomTrajectory(2, 4, 6, 14, {0.5, 1.25});
    Trajectory merged;
    EXPECT(full.addTrajectories({second}, &merged));
    EXPECT(merged.K() == 5);
    EXPECT_NEAR(merged.getMaxTime(), full.getMaxTime() + second.getMaxTime(), 1e-15);
    EXPECT_NEAR(merged.evaluate(full.getMaxTime() + 0.3, 0)[1], second.evaluate(0.3, 0)[1], 1e-13);
    EXPECT_NEAR(merged.evaluate(1.0, 2)[3], full.evaluate(1.0, 2)[3], 0.0);
    Trajectory bad;
    EXPECT(!full.addTrajectories({randomTrajectory(2, 3, 6, 15, {0.5, 1.25})}, &bad));
  }
  // offset: positions move, derivatives do not; too short an offset vector is refused
  {
    Trajectory moved = full;
    Eigen::VectorXd off(3);
    off[0] = 1.0; off[1] = -2.0; off[2] = 0.5;
    EXPECT(moved.offsetTrajectory(off));
    for (double t : probe) {
      const Eigen::VectorXd a = moved.evaluate(t, 0), b = full.evaluate(t, 0);
      for (int d = 0; d < 3; ++d) EXPECT_NEAR(a[d], b[d] + off[d], 1e-14);
      EXPECT_NEAR(a[3], b[3], 0.0);
      EXPECT_NEAR(moved.evaluate(t, 1)[1], full.evaluate(t, 1)[1], 0.0);
    }
    Eigen::VectorXd too_short(2);
    too_short[0] = too_short[1] = 0.0;
    EXPECT(!moved.offsetTrajectory(too_short));
  }
  // vertices at the segment boundaries
  {
    const Vertex v = full.getVertexAtTime(1.9, derivative_order::ACCELERATION);
    EXPECT(v.D() == 4 && v.getNumberOfConstraints() == 3);
    Eigen::VectorXd c;
    EXPECT(v.getConstraint(derivative_order::VELOCITY, &c));
    EXPECT_NEAR(c[2], full.evaluate(1.9, 1)[2], 0.0);
    EXPECT(full.getStartVertex(1).isEqualTol(full.getVertexAtTime(0.0, 1), 0.0));
    EXPECT(full.getGoalVertex(1).isEqualTol(full.getVertexAtTime(full.getMaxTime(), 1), 0.0));
    Vertex::Vector all;
    EXPECT(full.getVertices(derivative_order::JERK, &all));
    EXPECT(all.size() == 4 && all[2].getNumberOfConstraints() == 4);
    EXPECT(all[2].getConstraint(derivative_order::POSITION, &c));
    EXPECT_NEAR(c[0], full.evaluate(1.5 + 0.75, 0)[0], 0.0);
    Vertex::Vector pos, yaw;
    EXPECT(full.getVertices(derivative_order::ACCELERATION, derivative_order::VELOCITY, &pos, &yaw));
    EXPECT(pos.size() == 4 && yaw.size() == 4 && pos[1].D() == 3 && yaw[1].D() == 1);
    EXPECT(pos[1].getNumberOfConstraints() == 3 && yaw[1].getNumberOfConstraints() == 2);
    EXPECT(yaw[3].getConstraint(derivative_order::VELOCITY, &c));
    EXPECT_NEAR(c[0], full.evaluate(full.getMaxTime(), 1)[3], 0.0);
    // a 3-D trajectory has no yaw dimension to split off
    Vertex::Vector p3, y3;
    EXPECT(!randomTrajectory(2, 3, 6, 16, {1.0, 1.0}).getVertices(1, 1, &p3, &y3));
  }
}

// trajectory_sampling.h (reference src/trajectory_sampling.cpp): flat states of 3-, 4- and 6-dimensional trajectories.
static void quatToMatrix(const mav_msgs::Quaternion& q, double R[3][3]) {
  const double w = q.w, x = q.x, y = q.y, z = q.z;
  R[0][0] = 1 - 2 * (y * y + z * z); R[0][1] = 2 * (x * y - w * z);     R[0][2] = 2 * (x * z + w * y);
  R[1][0] = 2 * (x * y + w * z);     R[1][1] = 1 - 2 * (x * x + z * z); R[1][2] = 2 * (y * z - w * x);
  R[2][0] = 2 * (x * z - w * y);     R[2][1] = 2 * (y * z + w * x);     R[2][2] = 1 - 2 * (x * x + y * y);
}

static void testTrajectorySampling() {
  using mav_msgs::EigenTrajectoryPoint;
  const std::vector<double> times = {1.5, 0.75, 2.25};
  const Trajectory t4 = randomTrajectory(3, 4, 8, 21, times);
  {
    EigenTrajectoryPoint st;
    const double ts = 1.9;
    EXPECT(sampleTrajectoryAtTime(t4, ts, &st));
    for (int d = 0; d < 3; ++d) {
      EXPECT_NEAR(st.position_W[d], t4.evaluate(ts, 0)[d], 0.0);
      EXPECT_NEAR(st.velocity_W[d], t4.evaluate(ts, 1)[d], 0.0);
      EXPECT_NEAR(st.acceleration_W[d], t4.evaluate(ts, 2)[d], 0.0);
      EXPECT_NEAR(st.jerk_W[d], t4.evaluate(ts, 3)[d], 0.0);
      EXPECT_NEAR(st.snap_W[d], t4.evaluate(ts, 4)[d], 0.0);
    }
    const double yaw = t4.evaluate(ts, 0)[3];
    EXPECT_NEAR(std::remainder(st.getYaw() - yaw, 2.0 * M_PI), 0.0, 1e-14);
    EXPECT_NEAR(st.getYawRate(), t4.evaluate(ts, 1)[3], 0.0);
    EXPECT_NEAR(st.getYawAcc(), t4.evaluate(ts, 2)[3], 0.0);
    EXPECT(st.time_from_start_ns == static_cast<int64_t>(ts * 1e9));
    EXPECT(st.degrees_of_freedom == mav_msgs::DOF4);
    EXPECT(!sampleTrajectoryAtTime(t4, -0.1, &st));
    EXPECT(!sampleTrajectoryAtTime(t4, t4.getMaxTime() + 0.1, &st));
    EXPECT(!sampleTrajectoryAtTime(randomTrajectory(2, 2, 6, 22, {1.0, 1.0}), 0.5, &st));
    EXPECT(sampleSegmentAtTime(t4.segments()[1], 0.3, &st));
    EXPECT_NEAR(st.position_W[1], t4.segments()[1].evaluate(0.3, 0)[1], 0.0);
    EXPECT(!sampleSegmentAtTime(t4.segments()[1], 0.8, &st));
  }
  {  // range: the sample set of evaluateRange, one state per sample
    mav_msgs::EigenTrajectoryPointVector states, whole, by_duration;
    const double dt = 0.11;
    EXPECT(sampleTrajectoryInRange(t4, 0.4, 4.0, dt, &states));
    std::vector<Eigen::VectorXd> pos, acc;
    t4.evaluateRange(0.4, 4.0, dt, 0, &pos);
    t4.evaluateRange(0.4, 4.0, dt, 2, &acc);
    EXPECT(states.size() == pos.size() && !states.empty());
    for (size_t i = 0; i < states.size(); i += 5) {
      EXPECT_NEAR(states[i].position_W[2], pos[i][2], 0.0);
      EXPECT_NEAR(states[i].acceleration_W[0], acc[i][0], 0.0);
      EXPECT_NEAR(states[i].getYawAcc(), acc[i][3], 0.0);
      EXPECT(states[i].time_from_start_ns == static_cast<int64_t>((0.4 + dt * i) * 1e9));
    }
    EXPECT(sampleWholeTrajectory(t4, dt, &whole));
    EXPECT(sampleTrajectoryStartDuration(t4, 0.0, t4.getMaxTime(), dt, &by_duration));
    EXPECT(whole.size() == by_duration.size() && whole.size() > states.size());
    EXPECT(!sampleTrajectoryInRange(t4, 0.4, t4.getMaxTime() + 1.0, dt, &states));
  }
  {  // Matlab dump of the sampled states (io.h): one row per 0.01 s sample, 27 aligned columns
    // a private file (mkstemp): a fixed name in a shared temp directory may belong to another user or run
    const char* tmpdir = std::getenv("TMPDIR");
    std::string tmpl = std::string(tmpdir && *tmpdir ? tmpdir : "/tmp") + "/mtg_sampled_states_XXXXXX";
    const int fd = mkstemp(&tmpl[0]);
    EXPECT(fd >= 0);
    if (fd >= 0) close(fd);
    const std::string path = tmpl;
    EXPECT(sampledTrajectoryStatesToFile(path, t4));
    std::ifstream fin(path);
    std::string line;
    size_t rows = 0;
    double first_tm = -1.0, x_row10 = 0.0;
    size_t line_len = 0;
    while (std::getline(fin, line)) {
      std::istringstream ls(line);
      std::vector<double> vals;
      double v;
      while (ls >> v) vals.push_back(v);
      EXPECT(vals.size() == 27);
      if (rows == 0) {
        first_tm = vals[26];
        line_len = line.size();
      }
      EXPECT(line.size() == line_len);  // aligned columns
      if (rows == 10) x_row10 = vals[1];
      ++rows;
    }
    mav_msgs::EigenTrajectoryPointVector whole;
    EXPECT(sampleWholeTrajectory(t4, 0.01, &whole));
    EXPECT(rows == whole.size() && rows > 400);
    EXPECT_NEAR(first_tm, 1.5, 1e-12);
    EXPECT_NEAR(x_row10, whole[10].position_W[0], 1e-5 * (1.0 + std::abs(whole[10].position_W[0])));
    std::remove(path.c_str());
  }
  {  // 6-D: rotation vector in the last three dimensions; angular rates against finite differences of the rotation
    const Trajectory t6 = randomTrajectory(2, 6, 8, 23, {2.0, 1.5});
    const double ts = 1.3, hstep = 1e-5;
    EigenTrajectoryPoint s0, sp, sm;
    EXPECT(sampleTrajectoryAtTime(t6, ts, &s0));
    EXPECT(sampleTrajectoryAtTime(t6, ts + hstep, &sp));
    EXPECT(sampleTrajectoryAtTime(t6, ts - hstep, &sm));
    EXPECT(s0.degrees_of_freedom == mav_msgs::DOF6);
    double R0[3][3], Rp[3][3], Rm[3][3], W[3][3];
    quatToMatrix(s0.orientation_W_B, R0);
    quatToMatrix(sp.orientation_W_B, Rp);
    quatToMatrix(sm.orientation_W_B, Rm);
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        double acc = 0.0;
        for (int k = 0; k < 3; ++k) acc += (Rp[i][k] - Rm[i][k]) / (2 * hstep) * R0[j][k];  // dR/dt R^T
        W[i][j] = acc;
      }
    const double wn = std::sqrt(W[2][1] * W[2][1] + W[0][2] * W[0][2] + W[1][0] * W[1][0]);
    const double fd_tol = 1e-6 * (1.0 + wn);  // central differences of a fast rotation: ~1e-8 relative
    EXPECT_NEAR(s0.angular_velocity_W[0], W[2][1], fd_tol);
    EXPECT_NEAR(s0.angular_velocity_W[1], W[0][2], fd_tol);
    EXPECT_NEAR(s0.angular_velocity_W[2], W[1][0], fd_tol);
    EXPECT_NEAR(W[0][0], 0.0, fd_tol);  // skew symmetric: the quaternion is a unit rotation
    for (int d = 0; d < 3; ++d) {
      const double fd = (sp.angular_velocity_W[d] - sm.angular_velocity_W[d]) / (2 * hstep);
      EXPECT_NEAR(s0.angular_acceleration_W[d], fd, 1e-6 * (1.0 + std::abs(fd)));
    }
    // the rotation is the exponential of the sampled rotation vector: R phi = phi
    const Eigen::VectorXd p = t6.evaluate(ts, 0);
    for (int i = 0; i < 3; ++i)
      EXPECT_NEAR(R0[i][0] * p[3] + R0[i][1] * p[4] + R0[i][2] * p[5], p[3 + i], 1e-14);
    // near the zero rotation vector the series branch is used
    Segment tiny(2, 6);
    for (int d = 0; d < 6; ++d) {
      Eigen::VectorXd c(2);
      c[0] = d < 3 ? 1.0 : 1e-7 * (d - 2);
      c[1] = 0.25 * (d + 1);
      tiny[d] = Polynomial(2, c);
    }
    tiny.setTime(1.0);
    EigenTrajectoryPoint sz;
    EXPECT(sampleSegmentAtTime(tiny, 0.0, &sz));
    EXPECT_NEAR(sz.angular_velocity_W[0], 1.0, 1e-6);  // phi ~ 0: omega = dphi = (1.0, 1.25, 1.5)
    EXPECT_NEAR(sz.angular_velocity_W[2], 1.5, 1e-6);
  }
}

static void testLayoutOnly() {
  const Params& p = kParams[4];
  Vertex::Vector vertices = fixtureVertices(p);
  b200::Topology topo;
  b200::buildTopology(N, p.D, 4, &vertices, &topo);
  EXPECT(topo.n_all == 100 && topo.n_fixed == 19 && topo.n_free == 36);
  EXPECT(topo.kernel == 1);
}

// TwoVerticesSetup (test :743-787): Matlab golden coefficients.
static void testTwoVerticesSetup() {
  Vertex start(1), goal(1);
  for (int d = 0; d <= 4; ++d) start.addConstraint(d, 0.0);
  goal = start;
  goal.addConstraint(derivative_order::POSITION, 5.0);
  PolynomialOptimization<10> opt(1);
  Vertex::Vector vertices{start, goal};
  opt.setupFromVertices(vertices, {5.0 * 2.0 / 2.0}, derivative_order::SNAP);
  EXPECT(opt.solveLinear());
  Segment::Vector segments;
  opt.getSegments(&segments);
  checkPath(vertices, segments);
  const double matlab[10] = {-0.000000000000004, 0.000000000000004, -0.000000000000006, 0.000000000000003,
                             -0.000000000000001, 0.201600000000015, -0.134400000000012, 0.034560000000004,
                             -0.004032000000000, 0.000179200000000};
  const Eigen::VectorXd coeffs = segments[0].getPolynomialsRef()[0].getCoefficients();
  for (int i = 0; i < 10; ++i) EXPECT_NEAR(coeffs[i], matlab[i], 2e-14);
  EXPECT(opt.getNumberFreeConstraints() == 0 && opt.getNumberFixedConstraints() == 10);
}

// BASELINE config C1: the README example (reference README.md:105-139), v_max = a_max = 2.
static void testReadmeExample() {
  const int dimension = 3, derivative_to_optimize = derivative_order::SNAP;
  Vertex::Vector vertices;
  Vertex start(dimension), middle(dimension), end(dimension);
  start.makeStartOrEnd(Eigen::Vector3d(0, 0, 1), derivative_to_optimize);
  vertices.push_back(start);
  middle.addConstraint(derivative_order::POSITION, Eigen::Vector3d(1, 2, 3));
  vertices.push_back(middle);
  end.makeStartOrEnd(Eigen::Vector3d(2, 1, 5), derivative_to_optimize);
  vertices.push_back(end);
  std::vector<double> segment_times = estimateSegmentTimes(vertices, 2.0, 2.0);
  PolynomialOptimization<10> opt(dimension);
  opt.setupFromVertices(vertices, segment_times, derivative_to_optimize);
  EXPECT(opt.solveLinear());
  EXPECT(opt.getNumberFixedConstraints() == 11 && opt.getNumberFreeConstraints() == 4);
  Segment::Vector segments;
  opt.getSegments(&segments);
  checkPath(vertices, segments);
  // x-coefficients of both segments (SURVEY.md appendix B.8; reproduced by the CPU oracle, tests/test_oracle.py)
  const double s0[10] = {0, 0, 0, 0, 0, 1.339252819683e-02, -7.845546057916e-03, 1.954568943734e-03,
                         -2.392908039981e-04, 1.181394415329e-05};
  const double s1[10] = {1, 5.845294839088e-01, 3.552673810634e-03, -4.357594222295e-02, -1.385817588887e-03,
                         7.025146441719e-03, -4.564409065003e-03, 1.688225883678e-03, -2.991260062373e-04,
                         1.981495243341e-05};
  const Eigen::VectorXd c0 = segments[0][0].getCoefficients(), c1 = segments[1][0].getCoefficients();
  for (int i = 0; i < 10; ++i) {
    EXPECT_NEAR(c0[i], s0[i], 2e-12);  // survey values carry the reference-order rounding (~1e-11 relative)
    EXPECT_NEAR(c1[i], s1[i], 2e-12);
  }
  Trajectory trajectory;
  opt.getTrajectory(&trajectory);
  EXPECT_NEAR(trajectory.getMaxTime(), segment_times[0] + segment_times[1], 1e-12);
  const Eigen::VectorXd mid = trajectory.evaluate(segment_times[0], derivative_order::POSITION);
  EXPECT_NEAR(mid[0], 1.0, 1e-9);
  EXPECT_NEAR(mid[1], 2.0, 1e-9);
  EXPECT_NEAR(mid[2], 3.0, 1e-9);
}

// UnconstrainedLinearEstimateSegmentTimes (test :271-306)
static void testUnconstrainedLinear(const Params& p) {
  Vertex::Vector vertices = fixtureVertices(p);
  std::vector<double> times = estimateSegmentTimes(vertices, p.v_max, p.a_max);
  PolynomialOptimization<N> opt(p.D);
  EXPECT(opt.setupFromVertices(vertices, times, p.max_derivative));
  EXPECT(opt.solveLinear());
  EXPECT(opt.getLastStatus() == 0);
  Segment::Vector segments;
  opt.getSegments(&segments);
  Trajectory trajectory;
  opt.getTrajectory(&trajectory);
  EXPECT(trajectory.K() == p.num_segments && trajectory.D() == p.D && trajectory.N() == N);
  checkPath(vertices, segments);
  const double cost = opt.computeCost();
  const double numeric = costNumeric(trajectory, p.max_derivative, 0.001);
  EXPECT(std::abs(numeric - cost) <= numeric * 0.1);  // checkCost (:176-197)
  // updateSegmentTimes + solveLinear (the nonlinear optimiser's inner step): stretching time lowers cost
  std::vector<double> slower = times;
  for (double& t : slower) t *= 1.5;
  opt.updateSegmentTimes(slower);
  EXPECT(opt.solveLinear());
  EXPECT(opt.computeCost() < cost);
}

// ConstraintPacking (test :505-564)
static void testConstraintPacking(const Params& p) {
  Eigen::VectorXd lo = Eigen::VectorXd::Constant(p.D, -50.0), hi = Eigen::VectorXd::Constant(p.D, 50.0);
  for (size_t rep = 0; rep < 5; ++rep) {
    Vertex::Vector vertices = createRandomVertices(p.max_derivative, p.num_segments, lo, hi, 12345 + rep);
    std::vector<double> times = estimateSegmentTimes(vertices, 3.0, 5.0);
    PolynomialOptimization<N> opt(p.D);
    opt.setupFromVertices(vertices, times);
    opt.solveLinear();
    Segment::Vector segments;
    opt.getSegments(&segments);
    std::vector<Eigen::VectorXd> fixed, free_c;
    opt.getFixedConstraints(&fixed);
    opt.getFreeConstraints(&free_c);
    Eigen::MatrixXd M, A_inv, A, M_pinv;
    opt.getM(&M);
    opt.getAInverse(&A_inv);
    opt.getA(&A);
    opt.getMpinv(&M_pinv);
    EXPECT(int(fixed.size()) == p.D && int(free_c.size()) == p.D);
    for (int d = 0; d < p.D; ++d) {
      Eigen::VectorXd d_all(fixed[d].size() + free_c[d].size());
      for (int i = 0; i < fixed[d].size(); ++i) d_all[i] = fixed[d][i];
      for (int i = 0; i < free_c[d].size(); ++i) d_all[fixed[d].size() + i] = free_c[d][i];
      Eigen::VectorXd Md = M * d_all;
      Eigen::VectorXd pp = A_inv * Md;
      Eigen::VectorXd d_un = A * pp;
      Eigen::VectorXd d_re = M_pinv * d_un;
      for (int i = 0; i < d_all.size(); ++i) EXPECT_NEAR(d_all[i], d_re[i], 1e-6);
      for (size_t j = 0; j < segments.size(); ++j) {
        const Eigen::VectorXd p_seg = segments[j][d].getCoefficients(0);
        for (int k = 0; k < N; ++k) EXPECT_NEAR(p_seg[k], pp[j * N + k], 1e-6);
      }
    }
    // setFreeConstraints with the optimum reproduces the solution
    Segment::Vector again;
    opt.setFreeConstraints(free_c);
    opt.getSegments(&again);
    for (size_t j = 0; j < segments.size(); ++j)
      for (int d = 0; d < p.D; ++d) {
        const Eigen::VectorXd a = segments[j][d].getCoefficients(0), b = again[j][d].getCoefficients(0);
        for (int k = 0; k < N; ++k) EXPECT_NEAR(a[k], b[k], 1e-9 * (1.0 + std::abs(a[k])));
      }
  }
}

// The batch entry point returns, per problem, exactly what the single-problem object returns.
static void testBatchMatchesSingle() {
  const int D = 3, K = 8, B = 37;
  Eigen::VectorXd lo = Eigen::VectorXd::Constant(D, -10.0), hi = Eigen::VectorXd::Constant(D, 10.0);
  std::vector<Vertex::Vector> all_vertices;
  std::vector<std::vector<double> > all_times;
  for (int b = 0; b < B; ++b) {
    all_vertices.push_back(createRandomVertices(4, K, lo, hi, 1000 + b));
    all_times.push_back(estimateSegmentTimes(all_vertices.back(), 3.0, 5.0));
  }
  BatchPolynomialOptimization<N> batch(D);
  EXPECT(batch.setupFromVertices(all_vertices, all_times, derivative_order::SNAP));
  EXPECT(batch.solveLinear());
  EXPECT(batch.size() == size_t(B));
  std::vector<double> costs = batch.computeCosts();
  for (int b = 0; b < B; ++b) {
    EXPECT(batch.status()[b] == 0);
    PolynomialOptimization<N> opt(D);
    opt.setupFromVertices(all_vertices[b], all_times[b], derivative_order::SNAP);
    opt.solveLinear();
    Segment::Vector single, from_batch;
    opt.getSegments(&single);
    batch.getSegments(b, &from_batch);
    EXPECT(single.size() == from_batch.size());
    for (size_t j = 0; j < single.size(); ++j) EXPECT(single[j] == from_batch[j]);  // bitwise
    EXPECT_NEAR(costs[b], opt.computeCost(), 1e-12 * std::abs(costs[b]));
    if (b == 0) checkPath(all_vertices[b], from_batch);
  }
}

// Fused time allocation + solve equals estimateSegmentTimes() on the host followed by the batch solve.
// Batch widenings against the single-object mirror: Mellinger gradient = finite differences of computeCost() over
// re-solved objects (reference nonlinear_impl.h:286-364); evaluateRange == Trajectory::evaluateRange bit for bit.
static void testBatchMellingerAndRange() {
  const int K = 5, D = 3, B = 9;
  std::vector<Vertex::Vector> all_v;
  std::vector<std::vector<double> > all_t;
  for (int b = 0; b < B; ++b) {
    Eigen::VectorXd lo = Eigen::VectorXd::Constant(D, -10.0), hi = Eigen::VectorXd::Constant(D, 10.0);
    Vertex::Vector v = createRandomVertices(getHighestDerivativeFromN(N), K, lo, hi, 500 + b);
    all_t.push_back(estimateSegmentTimes(v, 3.0, 5.0));
    all_v.push_back(v);
  }
  BatchPolynomialOptimization<N> batch(D);
  batch.setupFromVertices(all_v, all_t, 4);
  batch.solveLinear();
  std::vector<double> cost, grad;
  batch.costGradientMellinger(&cost, &grad);
  for (int b = 0; b < B; ++b) {
    PolynomialOptimization<N> opt(D);
    opt.setupFromVertices(all_v[b], all_t[b], 4);
    opt.solveLinear();
    const double J = opt.computeCost();
    EXPECT_NEAR(cost[b], J, 1e-8 * std::abs(J));
    for (int n = 0; n < K; ++n) {
      std::vector<double> t = all_t[b];
      for (int i = 0; i < K; ++i) t[i] = std::max(0.1, i == n ? t[i] + 0.1 : t[i] - 0.1 / (K - 1.0));
      opt.updateSegmentTimes(t);
      opt.solveLinear();
      const double g = (opt.computeCost() - J) / 0.1;
      EXPECT_NEAR(grad[b * K + n], g, 1e-6 * std::max(std::abs(J), std::abs(g)));
    }
  }
  const std::vector<int> ders = {0, 1, 2, 3, 4};
  const int S = 64;
  std::vector<double> samples, st;
  std::vector<int32_t> ns;
  batch.evaluateRange(0.7, 9.0, 0.2, ders, S, &samples, &ns, &st);
  for (int b = 0; b < B; ++b) {
    Trajectory traj;
    batch.getTrajectory(b, &traj);
    for (size_t q = 0; q < ders.size(); ++q) {
      std::vector<Eigen::VectorXd> ref;
      std::vector<double> ref_t;
      traj.evaluateRange(0.7, 9.0, 0.2, ders[q], &ref, &ref_t);
      EXPECT(ns[b] == static_cast<int32_t>(ref.size()));
      for (size_t k = 0; k < ref.size() && k < size_t(S); ++k) {
        EXPECT(st[b * S + k] == ref_t[k]);
        for (int d = 0; d < D; ++d) EXPECT(samples[((size_t(b) * S + k) * ders.size() + q) * D + d] == ref[k][d]);
      }
    }
  }
}

static void testFusedWaypointSolve() {
  const int D = 3, K = 6, B = 19;
  Eigen::VectorXd lo = Eigen::VectorXd::Constant(D, -10.0), hi = Eigen::VectorXd::Constant(D, 10.0);
  std::vector<double> positions, times;
  for (int b = 0; b < B; ++b) {
    Vertex::Vector v = createRandomVertices(4, K, lo, hi, 7000 + b);
    std::vector<double> t = estimateSegmentTimesNfabian(v, 3.0, 5.0);
    times.insert(times.end(), t.begin(), t.end());
    for (const Vertex& vert : v) {
      Eigen::VectorXd p;
      vert.getConstraint(derivative_order::POSITION, &p);
      for (int d = 0; d < D; ++d) positions.push_back(p[d]);
    }
  }
  BatchPolynomialOptimization<N> a(D), b(D);
  EXPECT(a.setupFromWaypoints(B, K, positions.data(), times.data()));
  EXPECT(a.solveLinear());
  EXPECT(b.solveWaypointsNfabian(B, K, positions.data(), 3.0, 5.0));
  for (int i = 0; i < B * K; ++i) EXPECT_NEAR(b.segmentTimes()[i], times[i], 4e-16 * times[i]);
  double scale = 0.0, diff = 0.0;
  for (int i = 0; i < B * K * D * N; ++i) {
    scale = std::max(scale, std::abs(a.coefficients()[i]));
    diff = std::max(diff, std::abs(a.coefficients()[i] - b.coefficients()[i]));
  }
  EXPECT(diff <= 1e-12 * scale);
  for (int i = 0; i < B; ++i) EXPECT(b.status()[i] == 0);
}

int main(int argc, char** argv) {
  const bool cpu_only = argc > 1 && std::strcmp(argv[1], "--cpu-only") == 0;
  testValueTypesAndFixtures();
  testAMatrixInversion();
  testLayoutOnly();
  testYamlIo();
  testExtremaAndConversions();
  testTrajectoryReshaping();
  testTrajectorySampling();
  if (!cpu_only) {
    testTwoVerticesSetup();
    testReadmeExample();
    for (const Params& p : kParams) testUnconstrainedLinear(p);
    for (const Params& p : kParams) testConstraintPacking(p);
    testBatchMatchesSingle();
    testFusedWaypointSolve();
    testBatchMellingerAndRange();
  }
  std::printf("%s: %d checks, %d failures\n", cpu_only ? "cpu-only" : "full", g_checks, g_failures);
  return g_failures == 0 ? 0 : 1;
}
