//! The Cubic Spline interpolation strategy: coefficient construction (K6) and evaluation (K5) on
//! the device.  Boundary-condition enums as in the reference:
//! [`BoundaryCondition`] (whole dataset) > [`RowBoundary`] (one data row) > [`SingleBoundary`] (one side).
use std::{ffi::c_void, fmt::Debug};

use ndarray::{Array, ArrayBase, ArrayViewMut, Axis, Data, Dimension, Ix1, RemoveAxis};
use num_traits::{Euclid, Float};

use super::{eval_result, integral_result, DeviceTable1D, Interp1D, Interp1DDerivStrategy, Interp1DIntegralStrategy, Interp1DStrategy, Interp1DStrategyBuilder};
use crate::{ffi, BuilderError, InterpolateError, NdiElem};

/// element types usable with the CubicSpline strategy (float only, like the reference's `SplineNum`)
pub trait SplineNum: NdiElem + Float + Euclid {}
impl SplineNum for f32 {}
impl SplineNum for f64 {}

/// Boundary conditions for the whole dataset
#[derive(Debug, PartialEq, Eq)]
pub enum BoundaryCondition<T, D: Dimension> {
    /// first and second segment at a curve end are the same polynomial (default)
    NotAKnot,
    /// second derivative at the curve end is 0
    Natural,
    /// first derivative at the curve end is 0
    Clamped,
    /// periodic spline: first and last data element must be equal
    Periodic,
    /// individual conditions per data row and/or side; shape = data shape with axis 0 of length 1
    Individual(Array<RowBoundary<T>, D>),
}

/// Boundary condition for a single data row
#[derive(Debug, PartialEq, Eq, Clone)]
pub enum RowBoundary<T> {
    NotAKnot,
    Natural,
    Clamped,
    Mixed { left: SingleBoundary<T>, right: SingleBoundary<T> },
}

/// Boundary condition for one side of one data row
#[derive(Debug, PartialEq, Eq, Clone)]
pub enum SingleBoundary<T> {
    NotAKnot,
    /// same as `SecondDeriv(0.0)`
    Natural,
    /// same as `FirstDeriv(0.0)`
    Clamped,
    FirstDeriv(T),
    SecondDeriv(T),
}

impl<T, D: Dimension> Default for BoundaryCondition<T, D> {
    fn default() -> Self {
        Self::NotAKnot
    }
}

impl<T: SplineNum> SingleBoundary<T> {
    /// (kind code of `NDI_SB_*`, value)
    fn encode(&self) -> (i32, T) {
        match self {
            SingleBoundary::NotAKnot => (0, T::zero()),
            SingleBoundary::Natural => (1, T::zero()),
            SingleBoundary::Clamped => (2, T::zero()),
            SingleBoundary::FirstDeriv(v) => (3, *v),
            SingleBoundary::SecondDeriv(v) => (4, *v),
        }
    }
}

/// The CubicSpline 1d interpolation Strategy (Builder)
#[derive(Debug)]
pub struct CubicSpline<T, D: Dimension> {
    extrapolate: bool,
    boundary: BoundaryCondition<T, D>,
}

#[derive(Debug, Clone, Copy)]
enum Extrapolate {
    No = 0,
    Yes = 1,
    Periodic = 2,
}

/// The CubicSpline 1d interpolation Strategy (Implementation).
/// The coefficient arrays `a`, `b` live in the interpolator's device table; `spec` is the boundary
/// condition as the C ABI takes it, consumed by [`Interp1DStrategy::bind`] when the coefficients are built.
/// Same type parameters as the reference's `CubicSplineStrategy<Sd, D>`.
#[derive(Debug)]
pub struct CubicSplineStrategy<Sd, D>
where
    Sd: Data,
    D: Dimension + RemoveAxis,
{
    extrapolate: Extrapolate,
    spec: Option<BoundarySpec<Sd::Elem>>,
    _dim: std::marker::PhantomData<D>,
}

/// `bc_kind` plus, for `Individual`, one (kind, value) pair per column and side
#[derive(Debug)]
struct BoundarySpec<T> {
    kind: i32,
    lk: Vec<i32>,
    lv: Vec<T>,
    rk: Vec<i32>,
    rv: Vec<T>,
}

impl<T: SplineNum, D: Dimension + RemoveAxis> CubicSpline<T, D> {
    /// create a cubic-spline interpolation stratgy
    pub fn new() -> Self {
        Self { extrapolate: false, boundary: BoundaryCondition::NotAKnot }
    }

    /// does the strategy extrapolate? Default is `false`
    pub fn extrapolate(mut self, extrapolate: bool) -> Self {
        self.extrapolate = extrapolate;
        self
    }

    /// set the boundary condition
    pub fn boundary(mut self, boundary: BoundaryCondition<T, D>) -> Self {
        self.boundary = boundary;
        self
    }
}

impl<T: SplineNum, D: Dimension + RemoveAxis> Default for CubicSpline<T, D> {
    fn default() -> Self {
        Self::new()
    }
}

impl<Sd, Sx, D> Interp1DStrategyBuilder<Sd, Sx, D> for CubicSpline<Sd::Elem, D>
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    const MINIMUM_DATA_LENGHT: usize = 3;
    type FinishedStrat = CubicSplineStrategy<Sd, D>;

    fn build<Sx2>(self, _x: &ArrayBase<Sx2, Ix1>, data: &ArrayBase<Sd, D>) -> Result<CubicSplineStrategy<Sd, D>, BuilderError>
    where
        Sx2: Data<Elem = Sd::Elem>,
    {
        let (mut lk, mut rk, mut lv, mut rv) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
        let kind = match &self.boundary {
            BoundaryCondition::NotAKnot => 0,
            BoundaryCondition::Natural => 1,
            BoundaryCondition::Clamped => 2,
            BoundaryCondition::Periodic => 3,
            BoundaryCondition::Individual(bounds) => {
                let mut expect = data.raw_dim();
                expect[0] = 1;
                if expect != bounds.raw_dim() {
                    return Err(BuilderError::ShapeError(format!(
                        "Boundary conditions array has wrong shape. Expected: {expect:?}, got: {:?}",
                        bounds.raw_dim()
                    )));
                }
                for row in bounds.iter() {
                    let (l, r) = match row {
                        RowBoundary::NotAKnot => (SingleBoundary::NotAKnot, SingleBoundary::NotAKnot),
                        RowBoundary::Natural => (SingleBoundary::Natural, SingleBoundary::Natural),
                        RowBoundary::Clamped => (SingleBoundary::Clamped, SingleBoundary::Clamped),
                        RowBoundary::Mixed { left, right } => (left.clone(), right.clone()),
                    };
                    let ((a, b), (c, d)) = (l.encode(), r.encode());
                    lk.push(a);
                    lv.push(b);
                    rk.push(c);
                    rv.push(d);
                }
                4
            }
        };
        let extrapolate = if !self.extrapolate {
            Extrapolate::No
        } else if matches!(self.boundary, BoundaryCondition::Periodic) {
            Extrapolate::Periodic
        } else {
            Extrapolate::Yes
        };
        Ok(CubicSplineStrategy { extrapolate, spec: Some(BoundarySpec { kind, lk, lv, rk, rv }), _dim: std::marker::PhantomData })
    }
}

impl<Sd, Sx, D> Interp1DStrategy<Sd, Sx, D> for CubicSplineStrategy<Sd, D>
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    /// CubicSpline::calc_coefficients on the device (K6), once, with the uploaded tables
    fn bind(&mut self, data: &ArrayBase<Sd, D>, table: &mut DeviceTable1D) -> Result<(), BuilderError> {
        let Some(spec) = self.spec.take() else { return Ok(()) };
        let ptr_i = |v: &Vec<i32>| if v.is_empty() { std::ptr::null() } else { v.as_ptr() };
        let ptr_t = |v: &Vec<Sd::Elem>| if v.is_empty() { std::ptr::null() } else { v.as_ptr() as *const c_void };
        let mut bad_column = -1i64;
        let st = unsafe {
            ffi::ndi_interp1d_spline_build(table.0, spec.kind, ptr_i(&spec.lk), ptr_t(&spec.lv), ptr_i(&spec.rk), ptr_t(&spec.rv), &mut bad_column)
        };
        match st {
            ffi::NDI_OK => Ok(()),
            ffi::NDI_PERIODIC_MISMATCH => {
                let (first, last) = (data.index_axis(Axis(0), 0), data.index_axis(Axis(0), data.shape()[0] - 1));
                let msg = if data.ndim() == 1 {
                    format!("First: {:?}, last: {:?}", data.first().unwrap_or_else(|| unreachable!()), data.last().unwrap_or_else(|| unreachable!()))
                } else {
                    format!("First: {first:?}, last: {last:?}")
                };
                Err(BuilderError::ValueError(format!(
                    "for periodic boundary condition the first and last value must be equal. {msg}"
                )))
            }
            _ => panic!("ndi_interp1d_spline_build failed ({st}): {}", ffi::last_error()),
        }
    }

    fn interp_into(
        &self,
        interp: &Interp1D<Sd, Sx, D, Self>,
        mut target: ArrayViewMut<'_, Sd::Elem, D::Smaller>,
        x: Sx::Elem,
    ) -> Result<(), InterpolateError> {
        match target.as_slice_mut() {
            Some(out) => self.interp_batch_into(interp, &[x], out),
            None => {
                let mut scratch = Array::<Sd::Elem, _>::zeros(target.raw_dim());
                let res = self.interp_batch_into(interp, &[x], scratch.as_slice_mut().unwrap_or_else(|| unreachable!()));
                target.assign(&scratch);
                res
            }
        }
    }

    fn interp_batch_into(&self, interp: &Interp1D<Sd, Sx, D, Self>, xs: &[Sd::Elem], out: &mut [Sd::Elem]) -> Result<(), InterpolateError> {
        let mut first_bad = -1i64;
        let st = unsafe {
            ffi::ndi_interp1d_cubic(
                interp.table.0,
                xs.as_ptr() as *const c_void,
                xs.len() as i64,
                self.extrapolate as i32,
                out.as_mut_ptr() as *mut c_void,
                &mut first_bad,
            )
        };
        eval_result(st, xs, first_bad, "x")
    }
}

/// NOT in the reference: first and second derivative of the spline (scipy's `CubicSpline(x, nu)`)
impl<Sd, Sx, D> Interp1DDerivStrategy<Sd, Sx, D> for CubicSplineStrategy<Sd, D>
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    fn deriv_batch_into(&self, interp: &Interp1D<Sd, Sx, D, Self>, xs: &[Sd::Elem], out: &mut [Sd::Elem], order: i32) -> Result<(), InterpolateError> {
        assert!(order == 1 || order == 2, "CubicSpline derivative order must be 1 or 2, got {order}");
        let mut first_bad = -1i64;
        let st = unsafe {
            ffi::ndi_interp1d_cubic_deriv(
                interp.table.0,
                xs.as_ptr() as *const c_void,
                xs.len() as i64,
                self.extrapolate as i32,
                order,
                out.as_mut_ptr() as *mut c_void,
                &mut first_bad,
            )
        };
        eval_result(st, xs, first_bad, "x")
    }
}

/// NOT in the reference: the integral of the spline between two bounds (scipy's `CubicSpline.integrate`)
impl<Sd, Sx, D> Interp1DIntegralStrategy<Sd, Sx, D> for CubicSplineStrategy<Sd, D>
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    const INTEGRAL_KIND: i32 = ffi::NDI_INTEGRAL_CUBIC;
    fn integral_batch_into(&self, interp: &Interp1D<Sd, Sx, D, Self>, lo: &[Sd::Elem], hi: &[Sd::Elem], out: &mut [Sd::Elem]) -> Result<(), InterpolateError> {
        let (mut first_bad, mut bad_bound) = (-1i64, -1i32);
        let st = unsafe {
            ffi::ndi_interp1d_cubic_integral(
                interp.table.0,
                lo.as_ptr() as *const c_void,
                hi.as_ptr() as *const c_void,
                lo.len() as i64,
                self.extrapolate as i32,
                out.as_mut_ptr() as *mut c_void,
                &mut first_bad,
                &mut bad_bound,
            )
        };
        integral_result(st, lo, hi, first_bad, bad_bound)
    }
}
