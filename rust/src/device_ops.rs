//! The lowerable operator vocabulary beside src/ops.rs.  UNVERIFIED — see rust/README.md.
//!
//! Binary: the reference's uninstantiable enums `ops::{Add, …, Shr}` (src/ops.rs:23-129) get a device op code.
//! Unary: `Map` takes an opaque closure (src/view.rs:299-303, 880-889) which no device can run; the device accepts
//!   (a) the closed type-level set below (same idiom as ops.rs),
//!   (b) `Fold<B>` over `rows()` — the reference's only spelling of an axis reduction (src/view.rs:617-622, 250-252),
//!   (c) closures over `Sym<T>`, traced ONCE with symbolic values (`v.map_sym(|x| x * x + 1.0)`), as view.py::Sym does.
use std::rc::Rc;

use crate::ffi;
use crate::lower::Node;
use crate::ops::{Add, BitAnd, BitOr, BitXor, Div, Mul, Rem, Shl, Shr, Sub};

/// Element types with a device representation (mdim_dtype).  `usize` is U64, `bool` one byte.
pub trait DeviceElem: Copy + 'static {
    const DTYPE: i32;
    const IS_BOOL: bool = false;
    fn bits(self) -> u64;
}
macro_rules! device_elem {
    ($($t:ty => $d:expr, $bits:expr;)*) => { $(impl DeviceElem for $t { const DTYPE: i32 = $d; fn bits(self) -> u64 { ($bits)(self) } })* };
}
device_elem! {
    u8 => ffi::U8, |x: u8| x as u64;   i32 => ffi::I32, |x: i32| x as u32 as u64;   u32 => ffi::U32, |x: u32| x as u64;
    i64 => ffi::I64, |x: i64| x as u64;   u64 => ffi::U64, |x: u64| x;   usize => ffi::U64, |x: usize| x as u64;
    f32 => ffi::F32, |x: f32| x.to_bits() as u64;   f64 => ffi::F64, |x: f64| x.to_bits();
    i8 => ffi::I8, |x: i8| x as u8 as u64;   i16 => ffi::I16, |x: i16| x as u16 as u64;   u16 => ffi::U16, |x: u16| x as u64;
}
impl DeviceElem for bool { const DTYPE: i32 = ffi::U8; const IS_BOOL: bool = true; fn bits(self) -> u64 { self as u64 } }

/// `B: Binary<T, U>` of src/ops.rs:14-18 with a device op code.  `Pair` (src/ops.rs:25-29) has none: it yields a tuple VALUE.
pub trait DeviceBinary { const OP: i32; }
macro_rules! device_binary { ($($b:ty => $op:expr;)*) => { $(impl DeviceBinary for $b { const OP: i32 = $op; })* }; }
device_binary! { Add => ffi::ADD; Sub => ffi::SUB; Mul => ffi::MUL; Div => ffi::DIV; Rem => ffi::REM;
                 BitAnd => ffi::AND; BitOr => ffi::OR; BitXor => ffi::XOR; Shl => ffi::SHL; Shr => ffi::SHR; }

/// Closed unary vocabulary, uninstantiable like the binary enums.
pub enum Neg {} pub enum Not {} pub enum Abs {} pub enum Sqrt {}
pub struct Cast<T>(core::marker::PhantomData<T>);
pub trait DeviceUnary { const OP: i32; }
impl DeviceUnary for Neg { const OP: i32 = ffi::NEG; }
impl DeviceUnary for Not { const OP: i32 = ffi::NOT; }
impl DeviceUnary for Abs { const OP: i32 = ffi::ABS; }
impl DeviceUnary for Sqrt { const OP: i32 = ffi::SQRT; }

/// `|row| { let mut s = init; row.each(|x| s = B::call(s, x)); s }` — sequential, index order.
pub struct Fold<B, T> { pub init: T, _b: core::marker::PhantomData<B> }
impl<B, T> Fold<B, T> { pub fn new(init: T) -> Self { Fold { init, _b: core::marker::PhantomData } } }

pub fn binary_node(op: i32, a: &Rc<Node>, b: &Rc<Node>) -> Rc<Node> {
    let mut n = Node::new(ffi::BINARY, a.dtype);
    n.op = op; n.children = vec![a.clone(), b.clone()];
    Rc::new(n)
}
pub fn const_node(dtype: i32, bits: u64) -> Rc<Node> { let mut n = Node::new(ffi::CONST, dtype); n.imm = bits; Rc::new(n) }
pub fn unary_node(op: i32, a: &Rc<Node>, is_bool: bool) -> Rc<Node> {
    if op == ffi::NOT && is_bool { return binary_node(ffi::XOR, a, &const_node(a.dtype, 1)); }   // `!bool` is logical; the descriptor's NOT is bitwise
    let mut n = Node::new(ffi::UNARY, a.dtype);
    n.op = op; n.src_dtype = a.dtype; n.children = vec![a.clone()];
    Rc::new(n)
}
pub fn cast_node(a: &Rc<Node>, dtype: i32) -> Rc<Node> {
    if a.dtype == dtype { return a.clone(); }
    let mut n = Node::new(ffi::UNARY, dtype);
    n.op = ffi::CAST; n.src_dtype = a.dtype; n.children = vec![a.clone()];
    Rc::new(n)
}

/// A scalar element inside a traced `map_sym` closure.
#[derive(Clone)]
pub struct Sym<T: DeviceElem> { pub node: Rc<Node>, _t: core::marker::PhantomData<T> }
impl<T: DeviceElem> Sym<T> {
    pub fn of(node: Rc<Node>) -> Self { Sym { node, _t: core::marker::PhantomData } }
    pub fn lift(x: T) -> Self { Sym::of(const_node(T::DTYPE, x.bits())) }
    pub fn cast<U: DeviceElem>(self) -> Sym<U> { Sym::of(cast_node(&self.node, U::DTYPE)) }   // Rust `as`
    pub fn abs(self) -> Self { Sym::of(unary_node(ffi::ABS, &self.node, false)) }
    pub fn sqrt(self) -> Self { Sym::of(unary_node(ffi::SQRT, &self.node, false)) }
}
macro_rules! sym_op {
    ($($tr:ident $f:ident $op:expr;)*) => { $(
        impl<T: DeviceElem> core::ops::$tr for Sym<T> { type Output = Sym<T>; fn $f(self, o: Sym<T>) -> Sym<T> { Sym::of(binary_node($op, &self.node, &o.node)) } }
        impl<T: DeviceElem> core::ops::$tr<T> for Sym<T> { type Output = Sym<T>; fn $f(self, o: T) -> Sym<T> { Sym::of(binary_node($op, &self.node, &Sym::lift(o).node)) } }
    )* };
}
sym_op! { Add add ffi::ADD; Sub sub ffi::SUB; Mul mul ffi::MUL; Div div ffi::DIV; Rem rem ffi::REM; BitAnd bitand ffi::AND; BitOr bitor ffi::OR; BitXor bitxor ffi::XOR; }
impl<T: DeviceElem> core::ops::Neg for Sym<T> { type Output = Sym<T>; fn neg(self) -> Sym<T> { Sym::of(unary_node(ffi::NEG, &self.node, false)) } }
impl<T: DeviceElem> core::ops::Not for Sym<T> { type Output = Sym<T>; fn not(self) -> Sym<T> { Sym::of(unary_node(ffi::NOT, &self.node, T::IS_BOOL)) } }
