// dubins.h -- shortest Dubins curves for the front-end's one-shot (KinoAstar::asignShotTraj, front_end/include/front_end/kino_astar.h:237-266).
//
// The reference calls a third-party library for this: ompl::base::DubinsStateSpace (distance + interpolate) of OMPL, installed as
// ros-noetic-ompl (README.md:24; OMPL 1.5.x in ROS Noetic), absent from /root/reference and from this image.  This header restates the
// algorithm OMPL publishes for that class (src/ompl/base/spaces/src/DubinsStateSpace.cpp; L. E. Dubins 1957, with the closed forms of
// Shkel & Lumelsky 2001 on the normalised problem (0, 0, alpha) -> (d, 0, beta)): the six words are tried in the order
// LSL, RSR, RSL, LSR, RLR, LRL and a later word wins only if strictly shorter; a point of the curve is found by walking the three
// segments on the unit-radius problem and scaling by the turning radius.  Parity against OMPL's own arithmetic is UNPINNED (no OMPL
// here); the reference's callers of it (kino_astar.cpp) are pinned with this header standing in for OMPL (oracle/shim/ompl).
//
// Compiled for host and device (UALM_KHD) and templated on the trigonometry: TrigLibm (sin, cos, tan, atan2, acos of the C library,
// the default, what the host front-end and the reference pin use) or TrigDet (include/ualm_detmath.h, bit-identical on host and
// device).  max / min are spelled as std::max / std::min define them, so NaN operands pick the same side on both.
#pragma once
#include <float.h>
#include <math.h>

#include "../../include/ualm_detmath.h"

#if defined(__CUDACC__)
#define UALM_KHD __host__ __device__ __forceinline__
#else
#define UALM_KHD inline
#endif

struct TrigLibm {
    static UALM_KHD double sin(double x) { return ::sin(x); }
    static UALM_KHD double cos(double x) { return ::cos(x); }
    static UALM_KHD double tan(double x) { return ::tan(x); }
    static UALM_KHD double atan2(double y, double x) { return ::atan2(y, x); }
    static UALM_KHD double acos(double x) { return ::acos(x); }
};
struct TrigDet {
    static UALM_KHD double sin(double x) { return ualm_sin(x); }
    static UALM_KHD double cos(double x) { return ualm_cos(x); }
    static UALM_KHD double tan(double x) { return ualm_tan(x); }
    static UALM_KHD double atan2(double y, double x) { return ualm_atan2(y, x); }
    static UALM_KHD double acos(double x) { return ualm_acos(x); }
};

namespace ualm_dubins {

UALM_KHD double dmax(double a, double b) { return a < b ? b : a; }     // std::max
UALM_KHD double dmin(double a, double b) { return b < a ? b : a; }     // std::min

constexpr double kTwoPi = 2.0 * M_PI;
constexpr double kPi = M_PI;
constexpr double kEps = 1e-6;       // DUBINS_EPS
constexpr double kZero = -1e-7;     // DUBINS_ZERO

enum Seg { LEFT = 0, STRAIGHT = 1, RIGHT = 2 };

UALM_KHD double mod2pi(double x)
{
    if (x < 0 && x > kZero) return 0;
    double xm = x - kTwoPi * floor(x / kTwoPi);
    if (kTwoPi - xm < .5 * kEps) xm = 0.;
    return xm;
}

struct Path {
    Seg type[3] = {LEFT, STRAIGHT, LEFT};
    double len[3] = {0., DBL_MAX, 0.};     // an unset word is infinitely long
    UALM_KHD double length() const { return len[0] + len[1] + len[2]; }
    static UALM_KHD Path make(Seg a, Seg b, Seg c, double t, double p, double q)
    {
        Path r;
        r.type[0] = a; r.type[1] = b; r.type[2] = c;
        r.len[0] = t; r.len[1] = p; r.len[2] = q;
        return r;
    }
};

// the six words on the normalised problem
template <class T> UALM_KHD Path word_LSL(double d, double a, double b)
{
    const double ca = T::cos(a), sa = T::sin(a), cb = T::cos(b), sb = T::sin(b);
    const double tmp = 2. + d * d - 2. * (ca * cb + sa * sb - d * (sa - sb));
    if (tmp >= kZero) {
        const double theta = T::atan2(cb - ca, d + sa - sb);
        return Path::make(LEFT, STRAIGHT, LEFT, mod2pi(-a + theta), sqrt(dmax(tmp, 0.)), mod2pi(b - theta));
    }
    return Path();
}
template <class T> UALM_KHD Path word_RSR(double d, double a, double b)
{
    const double ca = T::cos(a), sa = T::sin(a), cb = T::cos(b), sb = T::sin(b);
    const double tmp = 2. + d * d - 2. * (ca * cb + sa * sb - d * (sb - sa));
    if (tmp >= kZero) {
        const double theta = T::atan2(ca - cb, d - sa + sb);
        return Path::make(RIGHT, STRAIGHT, RIGHT, mod2pi(a - theta), sqrt(dmax(tmp, 0.)), mod2pi(-b + theta));
    }
    return Path();
}
template <class T> UALM_KHD Path word_RSL(double d, double a, double b)
{
    const double ca = T::cos(a), sa = T::sin(a), cb = T::cos(b), sb = T::sin(b);
    const double tmp = d * d - 2. + 2. * (ca * cb + sa * sb - d * (sa + sb));
    if (tmp >= kZero) {
        const double p = sqrt(dmax(tmp, 0.));
        const double theta = T::atan2(ca + cb, d - sa - sb) - T::atan2(2., p);
        return Path::make(RIGHT, STRAIGHT, LEFT, mod2pi(a - theta), p, mod2pi(b - theta));
    }
    return Path();
}
template <class T> UALM_KHD Path word_LSR(double d, double a, double b)
{
    const double ca = T::cos(a), sa = T::sin(a), cb = T::cos(b), sb = T::sin(b);
    const double tmp = -2. + d * d + 2. * (ca * cb + sa * sb + d * (sa + sb));
    if (tmp >= kZero) {
        const double p = sqrt(dmax(tmp, 0.));
        const double theta = T::atan2(-ca - cb, d + sa + sb) - T::atan2(-2., p);
        return Path::make(LEFT, STRAIGHT, RIGHT, mod2pi(-a + theta), p, mod2pi(-b + theta));
    }
    return Path();
}
template <class T> UALM_KHD Path word_RLR(double d, double a, double b)
{
    const double ca = T::cos(a), sa = T::sin(a), cb = T::cos(b), sb = T::sin(b);
    const double tmp = .125 * (6. - d * d + 2. * (ca * cb + sa * sb + d * (sa - sb)));
    if (fabs(tmp) < 1.) {
        const double p = kTwoPi - T::acos(tmp);
        const double theta = T::atan2(ca - cb, d - sa + sb);
        const double t = mod2pi(a - theta + .5 * p);
        return Path::make(RIGHT, LEFT, RIGHT, t, p, mod2pi(a - b - t + p));
    }
    return Path();
}
template <class T> UALM_KHD Path word_LRL(double d, double a, double b)
{
    const double ca = T::cos(a), sa = T::sin(a), cb = T::cos(b), sb = T::sin(b);
    const double tmp = .125 * (6. - d * d + 2. * (ca * cb + sa * sb - d * (sa - sb)));
    if (fabs(tmp) < 1.) {
        const double p = kTwoPi - T::acos(tmp);
        const double theta = T::atan2(-ca + cb, d + sa - sb);
        const double t = mod2pi(-a + theta + .5 * p);
        return Path::make(LEFT, RIGHT, LEFT, t, p, mod2pi(b - a - t + p));
    }
    return Path();
}

template <class T> UALM_KHD Path shortest_normalised(double d, double a, double b)
{
    if (d < kEps && fabs(a - b) < kEps) return Path::make(LEFT, STRAIGHT, LEFT, 0., d, 0.);
    Path best = word_LSL<T>(d, a, b);
    double min_len = best.length();
    const Path cand[5] = {word_RSR<T>(d, a, b), word_RSL<T>(d, a, b), word_LSR<T>(d, a, b), word_RLR<T>(d, a, b), word_LRL<T>(d, a, b)};
    for (int k = 0; k < 5; k++) {
        const double len = cand[k].length();
        if (len < min_len) { min_len = len; best = cand[k]; }
    }
    return best;
}

// the shortest curve from (x, y, yaw) s1 to s2 with turning radius rho, in units of rho
template <class T = TrigLibm> UALM_KHD Path shortest(const double s1[3], const double s2[3], double rho)
{
    const double dx = s2[0] - s1[0], dy = s2[1] - s1[1];
    const double d = sqrt(dx * dx + dy * dy) / rho, th = T::atan2(dy, dx);
    return shortest_normalised<T>(d, mod2pi(s1[2] - th), mod2pi(s2[2] - th));
}
template <class T = TrigLibm> UALM_KHD double distance(const double s1[3], const double s2[3], double rho) { return rho * shortest<T>(s1, s2, rho).length(); }

// the point at fraction t in [0, 1] of the curve; yaw wrapped into [-pi, pi) like SO2StateSpace::enforceBounds
template <class T = TrigLibm> UALM_KHD void interpolate(const double from[3], const Path &path, double rho, double t, double out[3])
{
    double seg = t * path.length();
    double x = 0., y = 0., yaw = from[2];
    for (int i = 0; i < 3 && seg > 0; ++i) {
        const double v = dmin(seg, path.len[i]);
        const double phi = yaw;
        seg -= v;
        switch (path.type[i]) {
        case LEFT:
            x = x + T::sin(phi + v) - T::sin(phi); y = y - T::cos(phi + v) + T::cos(phi); yaw = phi + v;
            break;
        case RIGHT:
            x = x - T::sin(phi - v) + T::sin(phi); y = y + T::cos(phi - v) - T::cos(phi); yaw = phi - v;
            break;
        case STRAIGHT:
            x = x + v * T::cos(phi); y = y + v * T::sin(phi);
            break;
        }
    }
    out[0] = x * rho + from[0];
    out[1] = y * rho + from[1];
    double w = fmod(yaw, kTwoPi);
    if (w < -kPi) w += kTwoPi;
    else if (w >= kPi) w -= kTwoPi;
    out[2] = w;
}

} // namespace ualm_dubins
