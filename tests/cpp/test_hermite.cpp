// Shape-preserving cubics through include/ndarray_interp_b200.hpp (NOT in the reference): Pchip, Akima (akima and
// makima) and CubicHermite builders, evaluated with the spline's value, derivative and integral methods.  Expected
// values are exact: a plateau PCHIP keeps, a line Akima reproduces, and the cubic x^3 that CubicHermite reproduces from
// its own slopes.  Exit code = number of failed checks.
#include <cstdio>

#include "ndarray_interp_b200.hpp"

using namespace ndarray_interp;
using A = Array<double>;

static int failures = 0, checks = 0;
#define CHECK(cond)                                                                    \
    do { ++checks; if (!(cond)) { ++failures; std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); } } while (0)
template <class E, class F>
static bool throws(F&& f) {
    try { f(); } catch (const E&) { return true; } catch (...) { return false; }
    return false;
}

static void pchip() {
    // y = 0, 1, 1, 2: the knot slopes next to the plateau are 0, so the plateau stays flat and the rise monotone
    auto ip = Interp1DBuilder<double>(A{0.0, 1.0, 1.0, 2.0}).strategy(Pchip<double>::new_()).build();
    CHECK(ip.interp(1.5)[0] == 1.0 && ip.interp(1.25)[0] == 1.0);
    double prev = -1.0;
    bool monotone = true;
    for (int i = 0; i <= 300; ++i) { const double v = ip.interp(i * 0.01)[0]; monotone &= v >= prev; prev = v; }
    CHECK(monotone);
    CHECK(ip.interp_deriv(1.5)[0] == 0.0);
    CHECK(throws<InterpolateError>([&] { ip.interp(3.5); }));
    auto ex = Interp1DBuilder<double>(A{0.0, 1.0, 1.0, 2.0}).strategy(Pchip<double>::new_().extrapolate(true)).build();
    CHECK(std::isfinite(ex.interp(3.5)[0]));
    auto two = Interp1DBuilder<double>(A{1.0, 3.0}).strategy(Pchip<double>::new_()).build();    // n == 2: the line
    CHECK(std::fabs(two.interp(0.25)[0] - 1.5) <= 1e-15);
}

static void akima() {
    A x{0.0, 0.5, 1.5, 2.0, 3.5, 4.0}, y = A::zeros({6});
    for (size_t i = 0; i < 6; ++i) y[i] = 2.0 * x[i] + 1.0;
    for (const char* m : {"akima", "makima"}) {
        auto ip = Interp1DBuilder<double>(y).x(x).strategy(Akima<double>::new_().method(m)).build();
        CHECK(std::fabs(ip.interp(2.75)[0] - 6.5) <= 1e-12);
        CHECK(std::fabs(ip.interp_deriv(0.25)[0] - 2.0) <= 1e-12);
        CHECK(std::fabs(ip.integrate(0.0, 4.0)[0] - 20.0) <= 1e-12);
    }
    CHECK(throws<std::invalid_argument>([&] { Akima<double>::new_().method("spline"); }));
}

static void cubic_hermite() {
    A x{0.0, 1.0, 2.5, 3.0}, y = A::zeros({4}), d = A::zeros({4});
    for (size_t i = 0; i < 4; ++i) { y[i] = x[i] * x[i] * x[i]; d[i] = 3.0 * x[i] * x[i]; }
    auto ip = Interp1DBuilder<double>(y).x(x).strategy(CubicHermite<double>::new_(d).extrapolate(true)).build();
    CHECK(std::fabs(ip.interp(1.75)[0] - 1.75 * 1.75 * 1.75) <= 1e-12);
    CHECK(std::fabs(ip.interp_deriv(2.0)[0] - 12.0) <= 1e-12);
    CHECK(std::fabs(ip.interp_deriv(2.0, 2)[0] - 12.0) <= 1e-12);
    CHECK(std::fabs(ip.integrate(0.0, 2.0)[0] - 4.0) <= 1e-12);
    CHECK(throws<BuilderError>([&] { Interp1DBuilder<double>(y).x(x).strategy(CubicHermite<double>::new_(A{1.0, 2.0})).build(); }));
    auto f = Interp1DBuilder<float>(Array<float>{0.0f, 1.0f, 8.0f}).strategy(CubicHermite<float>::new_(Array<float>{0.0f, 3.0f, 12.0f})).build();
    CHECK(std::fabs(f.interp(1.5f)[0] - 3.375f) <= 1e-5f);
}

int main() {
    pchip();
    akima();
    cubic_hermite();
    std::printf("%d checks, %d failures\n", checks, failures);
    return failures;
}
