//! NOT in the reference: shape-preserving cubic interpolants whose knot slopes are computed on the device (K10) --
//! [`Pchip`] (scipy's `PchipInterpolator`), [`Akima`] (`Akima1DInterpolator`, method akima or makima) and
//! [`CubicHermite`] (`CubicHermiteSpline`, slopes given).  The coefficients take the spline's form, so evaluation,
//! derivatives and integrals run through the cubic-spline entry points of the C ABI.
use std::ffi::c_void;

use ndarray::{Array, ArrayBase, ArrayViewMut, Data, Dimension, Ix1, RemoveAxis};

use super::cubic_spline::SplineNum;
use super::{eval_result, integral_result, DeviceTable1D, Interp1D, Interp1DDerivStrategy, Interp1DIntegralStrategy, Interp1DStrategy, Interp1DStrategyBuilder};
use crate::{ffi, BuilderError, InterpolateError};

/// PCHIP: monotone data gives a monotone interpolant
#[derive(Debug, Default, Clone)]
pub struct Pchip {
    extrapolate: bool,
}

/// Akima's cubic; `makima` selects the modified weights
#[derive(Debug, Default, Clone)]
pub struct Akima {
    extrapolate: bool,
    makima: bool,
}

/// cubic Hermite interpolant with the given slopes `dydx` (shaped like the data)
#[derive(Debug)]
pub struct CubicHermite<T, D: Dimension> {
    extrapolate: bool,
    dydx: Array<T, D>,
}

/// The strategy the three builders produce: the slopes' kind, consumed by [`Interp1DStrategy::bind`]
#[derive(Debug)]
pub struct HermiteStrategy<Sd, D>
where
    Sd: Data,
    D: Dimension + RemoveAxis,
{
    extrapolate: i32,
    kind: i32,
    dydx: Option<Vec<Sd::Elem>>,
    _dim: std::marker::PhantomData<D>,
}

impl Pchip {
    pub fn new() -> Self {
        Self::default()
    }

    /// does the strategy extrapolate? Default is `false`
    pub fn extrapolate(mut self, extrapolate: bool) -> Self {
        self.extrapolate = extrapolate;
        self
    }
}

impl Akima {
    pub fn new() -> Self {
        Self::default()
    }

    /// does the strategy extrapolate? Default is `false`
    pub fn extrapolate(mut self, extrapolate: bool) -> Self {
        self.extrapolate = extrapolate;
        self
    }

    /// `"akima"` (default) or `"makima"`; panics on anything else
    pub fn method(mut self, method: &str) -> Self {
        assert!(method == "akima" || method == "makima", "Akima method must be \"akima\" or \"makima\", got {method:?}");
        self.makima = method == "makima";
        self
    }
}

impl<T: SplineNum, D: Dimension> CubicHermite<T, D> {
    pub fn new(dydx: Array<T, D>) -> Self {
        Self { extrapolate: false, dydx }
    }

    /// does the strategy extrapolate? Default is `false`
    pub fn extrapolate(mut self, extrapolate: bool) -> Self {
        self.extrapolate = extrapolate;
        self
    }
}

fn strategy<Sd: Data, D: Dimension + RemoveAxis>(kind: i32, extrapolate: bool, dydx: Option<Vec<Sd::Elem>>) -> HermiteStrategy<Sd, D> {
    HermiteStrategy { extrapolate: extrapolate as i32, kind, dydx, _dim: std::marker::PhantomData }
}

impl<Sd, Sx, D> Interp1DStrategyBuilder<Sd, Sx, D> for Pchip
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    const MINIMUM_DATA_LENGHT: usize = 2;
    type FinishedStrat = HermiteStrategy<Sd, D>;

    fn build<Sx2>(self, _x: &ArrayBase<Sx2, Ix1>, _data: &ArrayBase<Sd, D>) -> Result<HermiteStrategy<Sd, D>, BuilderError>
    where
        Sx2: Data<Elem = Sd::Elem>,
    {
        Ok(strategy(ffi::NDI_HERMITE_PCHIP, self.extrapolate, None))
    }
}

impl<Sd, Sx, D> Interp1DStrategyBuilder<Sd, Sx, D> for Akima
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    const MINIMUM_DATA_LENGHT: usize = 2;
    type FinishedStrat = HermiteStrategy<Sd, D>;

    fn build<Sx2>(self, _x: &ArrayBase<Sx2, Ix1>, _data: &ArrayBase<Sd, D>) -> Result<HermiteStrategy<Sd, D>, BuilderError>
    where
        Sx2: Data<Elem = Sd::Elem>,
    {
        let kind = if self.makima { ffi::NDI_HERMITE_MAKIMA } else { ffi::NDI_HERMITE_AKIMA };
        Ok(strategy(kind, self.extrapolate, None))
    }
}

impl<Sd, Sx, D> Interp1DStrategyBuilder<Sd, Sx, D> for CubicHermite<Sd::Elem, D>
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    const MINIMUM_DATA_LENGHT: usize = 2;
    type FinishedStrat = HermiteStrategy<Sd, D>;

    fn build<Sx2>(self, _x: &ArrayBase<Sx2, Ix1>, data: &ArrayBase<Sd, D>) -> Result<HermiteStrategy<Sd, D>, BuilderError>
    where
        Sx2: Data<Elem = Sd::Elem>,
    {
        if self.dydx.shape() != data.shape() {
            return Err(BuilderError::ShapeError(format!(
                "dydx has wrong shape. Expected: {:?}, got: {:?}",
                data.shape(),
                self.dydx.shape()
            )));
        }
        let dydx: Vec<Sd::Elem> = self.dydx.iter().cloned().collect();     // logical (C) order
        Ok(strategy(ffi::NDI_HERMITE_GIVEN, self.extrapolate, Some(dydx)))
    }
}

impl<Sd, Sx, D> Interp1DStrategy<Sd, Sx, D> for HermiteStrategy<Sd, D>
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    /// the knot slopes and coefficients on the device (K10), once, with the uploaded tables
    fn bind(&mut self, _data: &ArrayBase<Sd, D>, table: &mut DeviceTable1D) -> Result<(), BuilderError> {
        let ptr = self.dydx.as_ref().map_or(std::ptr::null(), |v| v.as_ptr() as *const c_void);
        let st = unsafe { ffi::ndi_interp1d_hermite_build(table.0, self.kind, ptr, 0) };
        match st {
            ffi::NDI_OK => Ok(()),
            _ => panic!("ndi_interp1d_hermite_build failed ({st}): {}", ffi::last_error()),
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
            ffi::ndi_interp1d_cubic(interp.table.0, xs.as_ptr() as *const c_void, xs.len() as i64, self.extrapolate,
                                    out.as_mut_ptr() as *mut c_void, &mut first_bad)
        };
        eval_result(st, xs, first_bad, "x")
    }
}

impl<Sd, Sx, D> Interp1DDerivStrategy<Sd, Sx, D> for HermiteStrategy<Sd, D>
where
    Sd: Data,
    Sd::Elem: SplineNum,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    fn deriv_batch_into(&self, interp: &Interp1D<Sd, Sx, D, Self>, xs: &[Sd::Elem], out: &mut [Sd::Elem], order: i32) -> Result<(), InterpolateError> {
        assert!(order == 1 || order == 2, "cubic derivative order must be 1 or 2, got {order}");
        let mut first_bad = -1i64;
        let st = unsafe {
            ffi::ndi_interp1d_cubic_deriv(interp.table.0, xs.as_ptr() as *const c_void, xs.len() as i64, self.extrapolate, order,
                                          out.as_mut_ptr() as *mut c_void, &mut first_bad)
        };
        eval_result(st, xs, first_bad, "x")
    }
}

impl<Sd, Sx, D> Interp1DIntegralStrategy<Sd, Sx, D> for HermiteStrategy<Sd, D>
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
            ffi::ndi_interp1d_cubic_integral(interp.table.0, lo.as_ptr() as *const c_void, hi.as_ptr() as *const c_void,
                                             lo.len() as i64, self.extrapolate, out.as_mut_ptr() as *mut c_void,
                                             &mut first_bad, &mut bad_bound)
        };
        integral_result(st, lo, hi, first_bad, bad_bound)
    }
}
