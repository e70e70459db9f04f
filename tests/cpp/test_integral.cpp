// Definite integrals through include/ndarray_interp_b200.hpp (NOT in the reference): Interp1D::integrate,
// interp_array_integral, interp_array_integral_into for Linear and CubicSpline.  Expected values are integrals of
// piecewise linear data and of a quadratic, which a cubic spline with matching end derivatives reproduces.
// Exit code = number of failed checks.
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

static void linear_integrals() {
    auto ip = Interp1D<double>::builder(A{0.0, 2.0, 2.0, 4.0}).build();       // x = 0, 1, 2, 3
    CHECK(ip.integrate(0.0, 3.0)[0] == 6.0);
    CHECK(ip.integrate(3.0, 0.0)[0] == -6.0);
    CHECK(ip.integrate(1.5, 1.5)[0] == 0.0);
    CHECK(ip.integrate(0.0, 1.0)[0] == 1.0);
    const double lo[] = {0.0, 1.0, 0.5}, hi[] = {2.0, 3.0, 0.5};
    auto ys = ip.interp_array_integral(ArrayView<double>{lo, {3}, {1}}, ArrayView<double>{hi, {3}, {1}});
    CHECK(ys[0] == 3.0 && ys[1] == 5.0 && ys[2] == 0.0);
    CHECK(throws<InterpolateError>([&] { ip.integrate(0.5, 3.5); }));
    auto ex = Interp1D<double>::builder(A{1.0, 2.0}).strategy(Linear<double>().extrapolate(true)).build();
    CHECK(ex.integrate(-1.0, 0.0)[0] == 0.5);
    auto iv = Interp1D<int32_t>::builder(Array<int32_t>{0, 10, 25}).build();
    CHECK(throws<std::invalid_argument>([&] { iv.integrate(0, 1); }));
}

static void cubic_integrals() {
    // y = x^2 with y'(0) = 0 and y'(4) = 8: the spline is the quadratic itself, its integral x^3 / 3
    A x{0.0, 1.0, 2.0, 3.0, 4.0}, y{0.0, 1.0, 4.0, 9.0, 16.0};
    auto bc = BoundaryCondition<double>::Individual({1}, {RowBoundary<double>::Mixed(SingleBoundary<double>::FirstDeriv(0.0),
                                                                                     SingleBoundary<double>::FirstDeriv(8.0))});
    auto ip = Interp1DBuilder<double>(y).x(x).strategy(CubicSpline<double>().boundary(bc).extrapolate(true)).build();
    const double lo[] = {0.0, 0.5, 1.0, 2.75, -1.0}, hi[] = {4.0, 1.5, 1.0, 0.25, 5.0};
    auto got = ip.interp_array_integral(ArrayView<double>{lo, {5}, {1}}, ArrayView<double>{hi, {5}, {1}});
    for (size_t i = 0; i < 5; ++i) CHECK(std::fabs(got[i] - (hi[i] * hi[i] * hi[i] - lo[i] * lo[i] * lo[i]) / 3.0) <= 1e-12);
    CHECK(ip.integrate(2.5, 2.5)[0] == 0.0);
    auto no = Interp1DBuilder<double>(y).x(x).strategy(CubicSpline<double>().boundary(bc)).build();
    CHECK(throws<InterpolateError>([&] { no.integrate(1.0, 4.5); }));
}

int main() {
    linear_integrals();
    cubic_integrals();
    std::printf("%d checks, %d failures\n", checks, failures);
    return failures;
}
