//! One dimensional interpolation along the first axis: `Interp1D`, `Interp1DBuilder`, the strategy
//! traits and the built-in strategies.  Same public surface as the reference's `interp1d` module;
//! the batch loop of `interp_array_into` is ONE kernel launch for the built-in strategies.
use std::{ffi::c_void, fmt::Debug};

use ndarray::{
    Array, Array1, ArrayBase, ArrayView, ArrayViewMut, ArrayViewMut1, Axis, Data, DimAdd, Dimension, Ix1,
    OwnedRepr, RemoveAxis,
};
use num_traits::cast;

use crate::{
    ffi,
    vector_extensions::{Monotonic, VectorExtensions},
    BuilderError, InterpolateError, NdiElem,
};

pub mod cubic_spline;
mod linear;
pub use linear::Linear;

/// NOT in the reference: derivatives of an interpolant, computed on the device (`ndi_interp1d_*_deriv`).  A trait of
/// its own, next to [`Interp1DStrategy`], so that the reference's strategy trait keeps exactly its items; implemented
/// by the built-in strategies ([`Linear`]: order 1, [`cubic_spline::CubicSplineStrategy`]: order 1 and 2).
pub trait Interp1DDerivStrategy<Sd, Sx, D>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
    Self: Sized,
{
    /// derivative of order `order` at every query of `xs` into the rows of `out` (`xs.len() * row length`), with the
    /// query handling and errors of [`Interp1DStrategy::interp_batch_into`].
    ///
    /// # panics
    /// When the strategy has no derivative of that order
    fn deriv_batch_into(&self, interpolator: &Interp1D<Sd, Sx, D, Self>, xs: &[Sd::Elem], out: &mut [Sd::Elem], order: i32) -> Result<(), InterpolateError>;
}

/// Owner of the opaque device handle (grid, data, spline coefficients in HBM).
/// Immutable after build, so it is shared freely between threads like the reference's `&self`.
#[derive(Debug)]
pub struct DeviceTable1D(pub(crate) *mut ffi::ndi_interp1d);
unsafe impl Send for DeviceTable1D {}
unsafe impl Sync for DeviceTable1D {}
impl Drop for DeviceTable1D {
    fn drop(&mut self) {
        unsafe { ffi::ndi_interp1d_destroy(self.0) };
    }
}

pub trait Interp1DStrategyBuilder<Sd, Sx, D>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension,
    Self: Sized,
{
    const MINIMUM_DATA_LENGHT: usize;
    type FinishedStrat: Interp1DStrategy<Sd, Sx, D>;

    /// initialize the strategy by validating data (signature of the reference trait, unchanged).
    /// Guarantees as in the reference: x strictly rising, `x.len() == data.shape()[0] >= MINIMUM_DATA_LENGHT`.
    /// Device-side preparation (spline coefficients) happens afterwards, in
    /// [`Interp1DStrategy::bind`], once the tables have been uploaded.
    fn build<Sx2>(
        self,
        x: &ArrayBase<Sx2, Ix1>,
        data: &ArrayBase<Sd, D>,
    ) -> Result<Self::FinishedStrat, BuilderError>
    where
        Sx2: Data<Elem = Sd::Elem>;
}

pub trait Interp1DStrategy<Sd, Sx, D>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension,
    Self: Sized,
{
    /// Interpolate at position `x` into `target` (shape = data shape without axis 0).
    fn interp_into(
        &self,
        interpolator: &Interp1D<Sd, Sx, D, Self>,
        target: ArrayViewMut<'_, Sd::Elem, D::Smaller>,
        x: Sx::Elem,
    ) -> Result<(), InterpolateError>;

    /// NOT in the reference trait.  Called once by [`Interp1DBuilder::build`] after
    /// [`Interp1DStrategyBuilder::build`], with the uploaded device copy of `(x, data)`; strategies that keep
    /// device-side state (the spline coefficients) create it here.  Provided: the default does nothing, so a
    /// strategy written against the reference's two trait methods compiles and runs unchanged
    /// (`examples/custom_strategy.rs`).
    fn bind(&mut self, _data: &ArrayBase<Sd, D>, _table: &mut DeviceTable1D) -> Result<(), BuilderError> {
        Ok(())
    }

    /// The batch loop.  `xs` and `out` are contiguous, `out` holds `xs.len()` rows.  The default
    /// is the reference's loop over `interp_into` (host code, for user strategies); the built-in
    /// strategies override it with one launch.
    fn interp_batch_into(
        &self,
        interpolator: &Interp1D<Sd, Sx, D, Self>,
        xs: &[Sd::Elem],
        out: &mut [Sd::Elem],
    ) -> Result<(), InterpolateError>
    where
        D: RemoveAxis,
    {
        let row_dim = interpolator.data.raw_dim().remove_axis(Axis(0));
        let w = row_dim.size();
        for (i, &x) in xs.iter().enumerate() {
            let row = ArrayViewMut::from_shape(row_dim.clone(), &mut out[i * w..(i + 1) * w])
                .unwrap_or_else(|_| unreachable!());
            self.interp_into(interpolator, row, x)?;
        }
        Ok(())
    }
}

/// One dimensional interpolator
#[derive(Debug)]
pub struct Interp1D<Sd, Sx, D, Strat>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension,
{
    /// x values are guaranteed to be strict monotonically rising
    pub(crate) x: ArrayBase<Sx, Ix1>,
    pub(crate) data: ArrayBase<Sd, D>,
    pub(crate) strategy: Strat,
    pub(crate) table: DeviceTable1D,
}

/// Create and configure a [Interp1D] Interpolator.
#[derive(Debug)]
pub struct Interp1DBuilder<Sd, Sx, D, Strat>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension,
{
    x: ArrayBase<Sx, Ix1>,
    data: ArrayBase<Sd, D>,
    strategy: Strat,
}

impl<Sd, D> Interp1D<Sd, OwnedRepr<Sd::Elem>, D, Linear>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    D: Dimension + RemoveAxis,
{
    /// Get the [Interp1DBuilder]
    pub fn builder(data: ArrayBase<Sd, D>) -> Interp1DBuilder<Sd, OwnedRepr<Sd::Elem>, D, Linear> {
        Interp1DBuilder::new(data)
    }
}

impl<Sd, Sx, Strat> Interp1D<Sd, Sx, Ix1, Strat>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    Strat: Interp1DStrategy<Sd, Sx, Ix1>,
{
    /// interpolation at one point when the data dimension is `Ix1`
    pub fn interp_scalar(&self, x: Sx::Elem) -> Result<Sd::Elem, InterpolateError> {
        let mut buffer = [cast::<f64, Sd::Elem>(0.0).unwrap_or_else(|| unimplemented!())];
        let view = ArrayViewMut1::from(buffer.as_mut_slice()).remove_axis(Axis(0));
        self.strategy.interp_into(self, view, x).map(|_| buffer[0])
    }
}

impl<Sd, Sx, D, Strat> Interp1D<Sd, Sx, D, Strat>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
    Strat: Interp1DStrategy<Sd, Sx, D>,
{
    /// interpolated values at `x`, one dimension smaller than the data
    pub fn interp(&self, x: Sx::Elem) -> Result<Array<Sd::Elem, D::Smaller>, InterpolateError> {
        let mut target = Array::zeros(self.data.raw_dim().remove_axis(Axis(0)));
        self.strategy.interp_into(self, target.view_mut(), x).map(|_| target)
    }

    /// like [`interp`](Interp1D::interp), into the provided buffer
    pub fn interp_into(&self, x: Sx::Elem, buffer: ArrayViewMut<'_, Sd::Elem, D::Smaller>) -> Result<(), InterpolateError> {
        self.strategy.interp_into(self, buffer, x)
    }

    /// interpolated values at all points in `xs`; output shape = `xs.shape() ++ data.shape()[1..]`
    pub fn interp_array<Sq, Dq>(
        &self,
        xs: &ArrayBase<Sq, Dq>,
    ) -> Result<Array<Sd::Elem, <Dq as DimAdd<D::Smaller>>::Output>, InterpolateError>
    where
        Sq: Data<Elem = Sd::Elem>,
        Dq: Dimension + DimAdd<D::Smaller>,
    {
        let mut shape = <Dq as DimAdd<D::Smaller>>::Output::zeros(xs.ndim() + self.data.ndim() - 1);
        for (dst, src) in shape.slice_mut().iter_mut().zip(xs.shape().iter().chain(self.data.shape()[1..].iter())) {
            *dst = *src;
        }
        let mut ys = Array::zeros(shape);
        self.interp_array_into(xs, ys.view_mut()).map(|_| ys)
    }

    /// like [`interp_array`](Interp1D::interp_array), into the provided buffer.
    /// One launch for the whole batch whatever the rank of `xs`.
    ///
    /// # panics
    /// When the provided buffer has the wrong shape
    pub fn interp_array_into<Sq, Dq>(
        &self,
        xs: &ArrayBase<Sq, Dq>,
        mut buffer: ArrayViewMut<'_, Sd::Elem, <Dq as DimAdd<D::Smaller>>::Output>,
    ) -> Result<(), InterpolateError>
    where
        Sq: Data<Elem = Sd::Elem>,
        Dq: Dimension + DimAdd<D::Smaller>,
    {
        let expect: Vec<usize> = xs.shape().iter().chain(self.data.shape()[1..].iter()).copied().collect();
        assert!(buffer.shape() == expect.as_slice(), "expected: {:?}, got: {:?}", expect, buffer.shape());
        let queries = xs.as_standard_layout();
        let q = queries.as_slice().unwrap_or_else(|| unreachable!());
        match buffer.as_slice_mut() {
            Some(out) => self.strategy.interp_batch_into(self, q, out),
            None => {
                // strided destination: evaluate into a contiguous scratch, then scatter on the host
                let mut scratch = Array::<Sd::Elem, _>::zeros(buffer.raw_dim());
                let res = self.strategy.interp_batch_into(self, q, scratch.as_slice_mut().unwrap_or_else(|| unreachable!()));
                buffer.assign(&scratch);
                res
            }
        }
    }

    /// Create a interpolator without any data validation (uploads the tables, skips the grid check).
    ///
    /// # Safety
    /// `x` strictly monotonic rising, `data.shape()[0] == x.len()`, `strategy` initialised for the data.
    pub fn new_unchecked(x: ArrayBase<Sx, Ix1>, data: ArrayBase<Sd, D>, strategy: Strat) -> Self {
        let table = upload(&x, &data, ffi::NDI_ASSUME_VALID).unwrap_or_else(|e| panic!("{e}"));
        Interp1D { x, data, strategy, table }
    }

    /// get `(x, data)` coordinate at given index
    pub fn index_point(&self, index: usize) -> (Sx::Elem, ArrayView<'_, Sd::Elem, D::Smaller>) {
        (self.x[index], self.data.index_axis(Axis(0), index))
    }

    /// The index of a known value left of, or at x (device search).
    pub fn get_index_left_of(&self, x: Sx::Elem) -> usize {
        self.x.get_lower_index(x)
    }

    pub fn is_in_range(&self, x: Sx::Elem) -> bool {
        self.x[0] <= x && x <= self.x[self.x.len() - 1]
    }
}

/// NOT in the reference: derivatives (see [`Interp1DDerivStrategy`]); shapes, errors and panics as the value methods
impl<Sd, Sx, D, Strat> Interp1D<Sd, Sx, D, Strat>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
    Strat: Interp1DStrategy<Sd, Sx, D> + Interp1DDerivStrategy<Sd, Sx, D>,
{
    /// derivative of order `order` at `x`, one dimension smaller than the data
    pub fn interp_deriv(&self, x: Sx::Elem, order: i32) -> Result<Array<Sd::Elem, D::Smaller>, InterpolateError> {
        let mut target = Array::zeros(self.data.raw_dim().remove_axis(Axis(0)));
        let out = target.as_slice_mut().unwrap_or_else(|| unreachable!());
        self.strategy.deriv_batch_into(self, &[x], out, order).map(|_| target)
    }

    /// derivatives at all points in `xs`; output shape = `xs.shape() ++ data.shape()[1..]`
    pub fn interp_array_deriv<Sq, Dq>(
        &self,
        xs: &ArrayBase<Sq, Dq>,
        order: i32,
    ) -> Result<Array<Sd::Elem, <Dq as DimAdd<D::Smaller>>::Output>, InterpolateError>
    where
        Sq: Data<Elem = Sd::Elem>,
        Dq: Dimension + DimAdd<D::Smaller>,
    {
        let mut shape = <Dq as DimAdd<D::Smaller>>::Output::zeros(xs.ndim() + self.data.ndim() - 1);
        for (dst, src) in shape.slice_mut().iter_mut().zip(xs.shape().iter().chain(self.data.shape()[1..].iter())) {
            *dst = *src;
        }
        let mut ys = Array::zeros(shape);
        self.interp_array_deriv_into(xs, ys.view_mut(), order).map(|_| ys)
    }

    /// like [`interp_array_deriv`](Interp1D::interp_array_deriv), into the provided buffer, which may have any
    /// layout (C order, Fortran order, permuted or reversed axes), as for
    /// [`interp_array_into`](Interp1D::interp_array_into):
    ///
    /// ```no_run
    /// use ndarray::{array, Array2, ShapeBuilder};
    /// use ndarray_interp_b200::interp1d::Interp1D;
    /// let ip = Interp1D::builder(array![[0.0, 1.0], [2.0, 4.0], [3.0, 9.0]]).build().unwrap();
    /// let xs = array![0.5, 1.5];
    /// let mut f_order = Array2::<f64>::zeros((2, 2).f());
    /// ip.interp_array_deriv_into(&xs, f_order.view_mut(), 1).unwrap();
    /// assert_eq!(f_order, array![[2.0, 3.0], [1.0, 5.0]]);
    /// ```
    ///
    /// # panics
    /// When the provided buffer has the wrong shape, or the strategy has no derivative of that order
    pub fn interp_array_deriv_into<Sq, Dq>(
        &self,
        xs: &ArrayBase<Sq, Dq>,
        mut buffer: ArrayViewMut<'_, Sd::Elem, <Dq as DimAdd<D::Smaller>>::Output>,
        order: i32,
    ) -> Result<(), InterpolateError>
    where
        Sq: Data<Elem = Sd::Elem>,
        Dq: Dimension + DimAdd<D::Smaller>,
    {
        let expect: Vec<usize> = xs.shape().iter().chain(self.data.shape()[1..].iter()).copied().collect();
        assert!(buffer.shape() == expect.as_slice(), "expected: {:?}, got: {:?}", expect, buffer.shape());
        let queries = xs.as_standard_layout();
        let q = queries.as_slice().unwrap_or_else(|| unreachable!());
        match buffer.as_slice_mut() {
            Some(out) => self.strategy.deriv_batch_into(self, q, out, order),
            None => {
                // strided destination: start from the caller's values, so rows after a failing query stay untouched
                // (standard layout: `to_owned` would keep an F-order or reversed buffer's strides)
                let mut scratch = Array::<Sd::Elem, _>::zeros(buffer.raw_dim());
                scratch.assign(&buffer);
                let res = self.strategy.deriv_batch_into(self, q, scratch.as_slice_mut().unwrap_or_else(|| unreachable!()), order);
                buffer.assign(&scratch);
                res
            }
        }
    }
}

/// upload of `(x, data)` as the views lie in memory (any strides: the library makes them dense on the device,
/// no `as_standard_layout()` copy on the host); the strict-rising check runs on the device unless skipped
pub(crate) fn upload<Sd, Sx, D>(x: &ArrayBase<Sx, Ix1>, data: &ArrayBase<Sd, D>, flags: u32) -> Result<DeviceTable1D, BuilderError>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension,
{
    let shape: Vec<i64> = data.shape().iter().map(|&s| s as i64).collect();
    let strides: Vec<i64> = data.strides().iter().map(|&s| s as i64).collect();   // ndarray strides are in elements
    let mut handle = std::ptr::null_mut();
    let st = unsafe {
        ffi::ndi_interp1d_create_strided(
            <Sd::Elem as NdiElem>::DTYPE,
            x.as_ptr() as *const c_void,          // first logical element, also for negative strides
            x.len() as i64,
            x.strides()[0] as i64,
            data.as_ptr() as *const c_void,
            shape.len() as i32,
            shape.as_ptr(),
            strides.as_ptr(),
            flags,
            &mut handle,
        )
    };
    match st {
        ffi::NDI_OK => Ok(DeviceTable1D(handle)),
        ffi::NDI_NOT_MONOTONIC => Err(BuilderError::Monotonic(ffi::last_error())),
        _ => panic!("ndi_interp1d_create failed ({st}): {}", ffi::last_error()),
    }
}

/// map an evaluation status to the reference's error / panic
pub(crate) fn eval_result<T: Debug>(st: ffi::ndi_status, xs: &[T], first_bad: i64, name: &str) -> Result<(), InterpolateError> {
    match st {
        ffi::NDI_OK => Ok(()),
        ffi::NDI_OUT_OF_BOUNDS => {
            let x = &xs[first_bad as usize];
            Err(InterpolateError::OutOfBounds(format!("{name} = {x:#?} is not in range")))
        }
        ffi::NDI_NAN_QUERY => unimplemented!("failed to convert NaN to usize"),
        _ => panic!("device evaluation failed ({st}): {}", ffi::last_error()),
    }
}

impl<Sd, D> Interp1DBuilder<Sd, OwnedRepr<Sd::Elem>, D, Linear>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    D: Dimension,
{
    /// Linear interpolation without extrapolation over the index of axis 0 unless configured otherwise.
    pub fn new(data: ArrayBase<Sd, D>) -> Self {
        let len = data.shape()[0];
        let x = Array1::from_iter((0..len).map(|n| cast(n).unwrap_or_else(|| unimplemented!("casting from usize to a number should always work"))));
        Interp1DBuilder { x, data, strategy: Linear::new() }
    }
}

impl<Sd, Sx, D, Strat> Interp1DBuilder<Sd, Sx, D, Strat>
where
    Sd: Data,
    Sd::Elem: NdiElem,
    Sx: Data<Elem = Sd::Elem>,
    D: Dimension + RemoveAxis,
    Strat: Interp1DStrategyBuilder<Sd, Sx, D>,
{
    /// custom x axis: same length and element type as the data, strict monotonic rising
    pub fn x<NewSx>(self, x: ArrayBase<NewSx, Ix1>) -> Interp1DBuilder<Sd, NewSx, D, Strat>
    where
        NewSx: Data<Elem = Sd::Elem>,
        Strat: Interp1DStrategyBuilder<Sd, NewSx, D>,
    {
        Interp1DBuilder { x, data: self.data, strategy: self.strategy }
    }

    /// Set the interpolation strategy
    pub fn strategy<NewStrat>(self, strategy: NewStrat) -> Interp1DBuilder<Sd, Sx, D, NewStrat>
    where
        NewStrat: Interp1DStrategyBuilder<Sd, Sx, D>,
    {
        Interp1DBuilder { x: self.x, data: self.data, strategy }
    }

    /// Validate input data and create the configured [Interp1D].
    /// Check order as in the reference: ndim, minimum length, monotonic, length match.
    pub fn build(self) -> Result<Interp1D<Sd, Sx, D, Strat::FinishedStrat>, BuilderError> {
        let Interp1DBuilder { x, data, strategy } = self;
        if data.ndim() < 1 {
            return Err(BuilderError::ShapeError("data dimension is 0, needs to be at least 1".into()));
        }
        if data.shape()[0] < Strat::MINIMUM_DATA_LENGHT {
            return Err(BuilderError::NotEnoughData(format!(
                "The chosen Interpolation strategy needs at least {} data points",
                Strat::MINIMUM_DATA_LENGHT
            )));
        }
        if !matches!(x.monotonic_prop(), Monotonic::Rising { strict: true }) {
            return Err(BuilderError::Monotonic("Values in the x axis need to be strictly monotonic rising".into()));
        }
        if x.len() != data.shape()[0] {
            return Err(BuilderError::ShapeError(format!(
                "Lengths of x and data axis need to match. Got x: {:}, data: {:}",
                x.len(),
                data.shape()[0],
            )));
        }
        let mut strategy = strategy.build(&x, &data)?;
        let mut table = upload(&x, &data, ffi::NDI_ASSUME_VALID)?;
        strategy.bind(&data, &mut table)?;
        Ok(Interp1D { x, data, strategy, table })
    }
}
