// Derivatives through include/ndarray_interp_b200.hpp (NOT in the reference): Interp1D::interp_deriv,
// interp_array_deriv, interp_array_deriv_into for Linear (order 1) and CubicSpline (order 1 and 2).
// Expected values are exact slopes of piecewise linear data and the derivatives of a quadratic, which a cubic spline
// with matching end derivatives reproduces.  Exit code = number of failed checks.
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

static void linear_slope() {
    auto ip = Interp1D<double>::builder(A{1.5, 2.0, 3.0, 4.0, 5.0, 7.0, 7.0, 8.0, 9.0, 10.5}).build();
    CHECK(ip.interp_deriv(0.5)[0] == 0.5);
    CHECK(ip.interp_deriv(4.0)[0] == 2.0);                   // a knot takes the interval to its right
    CHECK(ip.interp_deriv(9.0)[0] == 1.5);                   // the last knot: the last interval
    auto ys = ip.interp_array_deriv(A{0.25, 5.5, 8.5}.view());
    CHECK(ys[0] == 0.5 && ys[1] == 0.0 && ys[2] == 1.5);
    CHECK(throws<InterpolateError>([&] { ip.interp_deriv(9.5); }));
    CHECK(throws<std::invalid_argument>([&] { ip.interp_deriv(1.0, 2); }));
    auto ex = Interp1D<double>::builder(A{1.0, 2.0, 1.5}).strategy(Linear<double>().extrapolate(true)).build();
    CHECK(ex.interp_deriv(-1.0)[0] == 1.0 && ex.interp_deriv(3.0)[0] == -0.5);
    auto iv = Interp1D<int32_t>::builder(Array<int32_t>{0, 10, 25}).build();
    CHECK(iv.interp_deriv(1)[0] == 15);
}

static void cubic_derivatives() {
    // y = x^2 with y'(0) = 0 and y'(4) = 8: the spline is the quadratic itself
    A x{0.0, 1.0, 2.0, 3.0, 4.0}, y{0.0, 1.0, 4.0, 9.0, 16.0};
    auto bc = BoundaryCondition<double>::Individual({1}, {RowBoundary<double>::Mixed(SingleBoundary<double>::FirstDeriv(0.0),
                                                                                     SingleBoundary<double>::FirstDeriv(8.0))});
    auto ip = Interp1DBuilder<double>(y).x(x).strategy(CubicSpline<double>().boundary(bc).extrapolate(true)).build();
    const double q[] = {0.0, 0.5, 1.0, 2.75, 4.0, 5.0};
    auto d1 = ip.interp_array_deriv(ArrayView<double>{q, {6}, {1}}, 1);
    auto d2 = ip.interp_array_deriv(ArrayView<double>{q, {6}, {1}}, 2);
    for (size_t i = 0; i < 6; ++i) {
        CHECK(std::fabs(d1[i] - 2.0 * q[i]) <= 1e-12);
        CHECK(std::fabs(d2[i] - 2.0) <= 1e-12);
    }
    CHECK(std::fabs(ip.interp_deriv(1.5)[0] - 3.0) <= 1e-12);
    Array<double> buf = Array<double>::zeros({2});
    ip.interp_array_deriv_into(ArrayView<double>{q + 1, {2}, {1}}, buf.view_mut(), 2);
    CHECK(std::fabs(buf[0] - 2.0) <= 1e-12 && std::fabs(buf[1] - 2.0) <= 1e-12);
    CHECK(throws<std::invalid_argument>([&] { ip.interp_deriv(1.0, 3); }));
    auto no = Interp1DBuilder<double>(y).x(x).strategy(CubicSpline<double>().boundary(bc)).build();
    CHECK(throws<InterpolateError>([&] { no.interp_deriv(4.5); }));
    auto f = Interp1DBuilder<float>(Array<float>{0.0f, 1.0f, 4.0f, 9.0f, 16.0f}).x(Array<float>{0.0f, 1.0f, 2.0f, 3.0f, 4.0f})
                 .strategy(CubicSpline<float>().boundary(BoundaryCondition<float>::Individual({1}, {RowBoundary<float>::Mixed(
                     SingleBoundary<float>::FirstDeriv(0.0f), SingleBoundary<float>::FirstDeriv(8.0f))})))
                 .build();
    CHECK(std::fabs(f.interp_deriv(2.5f)[0] - 5.0f) <= 1e-5f && std::fabs(f.interp_deriv(2.5f, 2)[0] - 2.0f) <= 1e-4f);
}

int main() {
    linear_slope();
    cubic_derivatives();
    std::printf("%d checks, %d failures\n", checks, failures);
    return failures;
}
