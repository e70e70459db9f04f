//! Linear interpolation strategy: K3 `interp1d_linear_kernel` behind `ndi_interp1d_linear`.
use std::ffi::c_void;

use ndarray::{ArrayBase, ArrayViewMut, Data, Dimension, Ix1, RemoveAxis};

use super::{eval_result, Interp1D, Interp1DDerivStrategy, Interp1DStrategy, Interp1DStrategyBuilder};
use crate::{ffi, BuilderError, InterpolateError, NdiElem};

/// Linear Interpolation Strategy
#[derive(Debug)]
pub struct Linear {
    extrapolate: bool,
}

impl Linear {
    /// create a linear interpolation stratgy
    pub fn new() -> Self {
        Self { extrapolate: false }
    }

    /// does the strategy extrapolate? Default is `false`
    pub fn extrapolate(mut self, extrapolate: bool) -> Self {
        self.extrapolate = extrapolate;
        self
    }
}

impl Default for Linear {
    fn default() -> Self {
        Self::new()
    }
}

impl<Sd, Sx, D> Interp1DStrategyBuilder<Sd, Sx, D> for Linear
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    const MINIMUM_DATA_LENGHT: usize = 2;
    type FinishedStrat = Linear;

    fn build<Sx2>(self, _x: &ArrayBase<Sx2, Ix1>, _data: &ArrayBase<Sd, D>) -> Result<Linear, BuilderError>
    where
        Sx2: Data<Elem = Sd::Elem>,
    {
        Ok(self)
    }
}

impl<Sd, Sx, D> Interp1DStrategy<Sd, Sx, D> for Linear
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    fn interp_into(
        &self,
        interpolator: &Interp1D<Sd, Sx, D, Self>,
        mut target: ArrayViewMut<'_, Sd::Elem, D::Smaller>,
        x: Sx::Elem,
    ) -> Result<(), InterpolateError> {
        // one query through the batched launch (latency path of the C ABI)
        match target.as_slice_mut() {
            Some(out) => self.interp_batch_into(interpolator, &[x], out),
            None => {
                let mut scratch = ndarray::Array::<Sd::Elem, _>::zeros(target.raw_dim());
                let res = self.interp_batch_into(interpolator, &[x], scratch.as_slice_mut().unwrap_or_else(|| unreachable!()));
                target.assign(&scratch);
                res
            }
        }
    }

    fn interp_batch_into(&self, interpolator: &Interp1D<Sd, Sx, D, Self>, xs: &[Sd::Elem], out: &mut [Sd::Elem]) -> Result<(), InterpolateError> {
        let mut first_bad = -1i64;
        let st = unsafe {
            ffi::ndi_interp1d_linear(
                interpolator.table.0,
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

/// NOT in the reference: the slope `(y[i+1] - y[i]) / (x[i+1] - x[i])` of each query's interval
impl<Sd, Sx, D> Interp1DDerivStrategy<Sd, Sx, D> for Linear
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
{
    fn deriv_batch_into(&self, interpolator: &Interp1D<Sd, Sx, D, Self>, xs: &[Sd::Elem], out: &mut [Sd::Elem], order: i32) -> Result<(), InterpolateError> {
        assert!(order == 1, "Linear has only a first derivative, got order {order}");
        let mut first_bad = -1i64;
        let st = unsafe {
            ffi::ndi_interp1d_linear_deriv(
                interpolator.table.0,
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
