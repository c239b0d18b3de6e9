"""tools/minijl — the Julia-subset interpreter that executes the unmodified reference sources for the fixtures
(tests/golden/make_ref_fixtures.py).  It is test infrastructure, and a wrong interpreter would pin the oracle to the wrong
thing, so its semantics are tested here on the Julia features the reference's MCMC path relies on: operator precedence,
1-based column-major arrays, copies vs views, multiple dispatch incl. parametric and functor methods, keyword arguments,
closures, ranges, control flow, string interpolation, the scripted `rand`, and Julia's Float64 printing."""
import io
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from minijl.interp import Interp, JlError, jl_float  # noqa: E402


def run(src):
    out = io.StringIO()
    it = Interp(stdout=out, stderr=io.StringIO())
    val = it.run_string(src)
    return val, out.getvalue(), it


def ev(src):
    return run(src)[0]


def test_arithmetic_and_precedence():
    assert ev("-2^2") == -4 and ev("2^3^2") == 512 and ev("-1/2*4.0*3") == -6.0
    assert ev("1:3 == 1:3") is True
    assert ev("7 % 3") == 1 and ev("-7 % 3") == -1                    # rem, sign of the dividend
    assert ev("3/2") == 1.5 and ev("1/0") == float("inf")
    assert ev("x = 3.0; x^2") == 9.0 and ev("x = 1.0000000001; x^2 == x*x") is True     # literal_pow
    assert ev("2π") == 2 * np.pi and ev("3π/8") == 3 * np.pi / 8
    assert ev("a = 5; a < 6 && a > 4 || error(\"no\")") is True
    assert ev("true ? 1 : 2") == 1 and ev("x = 4; x > 5 ? 1 : x > 3 ? 2 : 3") == 2
    assert ev("min(π, max(0.0, 4.0))") == np.pi and ev("1 < 2 < 3") is True
    with pytest.raises(JlError):
        ev("1 && true")                                                # non-boolean in a boolean context


def test_arrays_are_one_based_column_major_and_slices_copy():
    v, _, it = run("""
A = zeros(3, 4)
for j in 1:4
  A[:, j] = [1.0*j; 10.0*j; 100.0*j]
end
col = A[:, 2]          # a copy
col[1] = -1.0
w = view(A, :, 3)      # a view
w[1] = 77.0
B = reshape(A, 1, :)   # column-major order
(A[1, 2], A[1, 3], B[1, 4], A[end, end], A[2], length(A), size(A, 2))
""")
    assert v == (2.0, 77.0, 2.0, 400.0, 10.0, 12, 4)
    assert ev("x = [1, 2, 3, 4, 5, 6]; x[1:2:end]").tolist() == [1, 3, 5]
    assert ev("x = [10, 20, 30]; x[end]") == 30
    assert ev("cumsum([1.0 2.0; 3.0 4.0], dims=2)").tolist() == [[1.0, 3.0], [3.0, 7.0]]
    assert ev("sum([1.0 2.0; 3.0 4.0], dims=2)").tolist() == [[3.0], [7.0]]
    assert ev("hcat(1, transpose([2.0, 3.0]), 4.0)").tolist() == [[1.0, 2.0, 3.0, 4.0]]
    assert ev("[1.0 0.0; 0.0 2.0] * [3.0; 4.0]").tolist() == [3.0, 8.0]
    assert ev("hcat(map(j -> [j; 2j], 1:3)...)").tolist() == [[1, 2, 3], [2, 4, 6]]
    assert ev("v = [1.0, 2.0]; w = v; w[1] = 9.0; v[1]") == 9.0          # arrays are references
    assert ev("v = [1.0, 2.0]; w = copy(v); w[1] = 9.0; v[1]") == 1.0
    with pytest.raises(JlError):
        ev("x = [1, 2, 3]; x[4]")
    with pytest.raises(JlError):
        ev("x = [1, 2, 3]; x[0]")
    with pytest.raises(JlError):
        ev("[1.0, 2.0] + 1.0")                                         # no implicit broadcasting


def test_multiple_dispatch_functors_and_parametric_methods():
    v, out, _ = run("""
abstract type Shape end
struct Circle <: Shape
  r::Float64
end
struct Square <: Shape
  a::Float64
end
area(s::Shape) = error("not implemented")
area(c::Circle) = π * c.r^2
area(s::Square) = s.a^2
(c::Circle)(k::Real) = Circle(k * c.r)
(::Shape)(::Real) = error("abstract")
describe(x::Integer) = "integer"
describe(x::Real) = "real"
describe(x::AbstractVector) = "vector"
describe(x) = "any"
mutable struct Box{T,N}
  value::T
  count::N
end
bump!(b::Box) = (b.count += 1; "scalar box")
bump!(b::Box{<:Vector}) = (b.count += 1; "vector box")
Circle(c::Circle) = Circle(c.r)          # an outer constructor next to the default one
f(x; scale::Real = 2.0, shift = 0) = scale * x + shift
(area(Circle(2)(0.5)), area(Square(3.0)), describe(1), describe(1.5), describe([1.0]), describe("s"),
 bump!(Box(1.0, 0)), bump!(Box([1.0, 2.0], 0)), Circle(Circle(4.0)).r, f(3.0), f(3.0; scale = 1, shift = 1))
""")
    assert v == (np.pi, 9.0, "integer", "real", "vector", "any", "scalar box", "vector box", 4.0, 6.0, 4.0)
    with pytest.raises(JlError, match="no method matching"):
        ev("g(x::Int) = 1; g(1.5)")
    with pytest.raises(JlError, match="immutable"):
        ev("struct P\n x::Float64\nend\np = P(1.0); p.x = 2.0")


def test_closures_loops_and_scope():
    assert ev("""
function counter()
  n = 0
  inc = () -> (n += 1; n)
  inc(); inc()
  return n
end
counter()""") == 2
    assert ev("""
function f()
  s = 0
  for i = 1:10
    if i % 2 == 0; continue; end
    if i > 7; break; end
    s += i
  end
  k = 0
  while true
    k += 1
    k >= 3 && break
  end
  return (s, k)
end
f()""") == (16, 3)
    assert ev("[i*i for i in 1:5 if i != 3]").tolist() == [1, 4, 16, 25]
    assert ev("a, b = if true\n 1, 2\n else\n 3, 4\n end; a + b") == 3
    assert ev("x = 10; function g(); x = 1; x; end; g(); x") == 10          # a function's assignment is local
    assert ev("acc = Any[]; foreach(v -> push!(acc, 2v), [1, 2, 3]); acc") == [2, 4, 6]


def test_strings_printing_and_julia_float_text():
    _, out, _ = run('x = [1.0, 2.5e-7, 1.0e21]; n = 3; println("<r> = $(x) $n $(n/2)"); println("AR     =   ", 0.3016666666666667)')
    assert out == "<r> = [1.0, 2.5e-7, 1.0e21] 3 1.5\nAR     =   0.3016666666666667\n"
    for x, s in ((500.0, "500.0"), (1e-5, "1.0e-5"), (0.0001, "0.0001"), (123456.7, "123456.7"), (1234567.0, "1.234567e6"),
                 (-0.0, "-0.0"), (float("inf"), "Inf"), (1e22, "1.0e22"), (0.1 + 0.2, "0.30000000000000004")):
        assert jl_float(x) == s


def test_scripted_rand_shadows_the_builtin_and_an_unscripted_rand_fails():
    with pytest.raises(JlError, match="scripted"):
        ev("rand()")
    v = ev("""
const TAPE = Any[0.25, 0.5, 0.75, 0.1]
rand() = popfirst!(TAPE)
rand(d::Uniform) = d.a + (d.b - d.a) * rand()
rand(r::UnitRange) = r[1 + floor(Int, rand() * length(r))]
rand(::Type{Bool}) = rand() < 0.5
(rand(1:8), rand(Uniform(-2.0, 2.0)), rand(), rand(Bool))""")
    assert v == (3, 0.0, 0.75, True)


def test_the_reference_energy_functions_reproduce_the_survey_kat():
    """End to end on the unmodified inc/eap_chain.jl (when the reference tree is there): SURVEY §8c's n=5 known answers."""
    ref = os.environ.get("POLYMC_REFERENCE_DIR")
    if not ref or not os.path.isdir(os.path.join(ref, "inc")):
        pytest.skip("needs the reference sources: set POLYMC_REFERENCE_DIR")
    v = ev("""
const TAPE = Any[]
rand() = popfirst!(TAPE)
rand(d::Uniform) = d.a + (d.b - d.a) * rand()
rand(d::Uniform, n::Int) = [rand(d) for i in 1:n]
include(""" + json.dumps(os.path.join(ref, "inc", "eap_chain.jl")) + """)
function kat()
  p = Dict{String,Any}()
  p["num-monomers"] = 5; p["mlen"] = 1.5; p["E0"] = 2.0; p["K1"] = 1.0; p["K2"] = 0.25; p["mu"] = 0.5
  p["kT"] = 1.0; p["Fz"] = 0.7; p["Fx"] = 0.3; p["chain-type"] = "dielectric"; p["energy-type"] = "interacting"
  for x in [0.1, 1.3, 2.9, 4.4, 5.9]
    push!(TAPE, x / (2*π))
  end
  for x in [0.4, 1.1, 1.7, 2.3, 2.9]
    push!(TAPE, x / π)
  end
  c = EAPChain(p)
  return (c.U, c.Ω, U_Ising(c))
end
kat()""")
    assert v[0] == pytest.approx(-5.804047873024686, rel=1e-13)
    assert v[1] == pytest.approx(-2.7903233230265996, rel=1e-13)


# ---- ccall (minijl/ffi.py): marshalling checked against a C library compiled on the spot -------------------------------
FFI_C = r"""
#include <stdint.h>
#include <string.h>
typedef struct { double a; double b; int64_t n; int32_t k; int32_t flag; double tail; } rec_t;   /* 40 bytes */
static char msg[64];
int32_t rec_sum(const rec_t* r, int64_t count, double* out) {     /* array of isbits structs in, one double out */
  double s = 0; for (int64_t i = 0; i < count; ++i) s += r[i].a + 10 * r[i].b + 100 * r[i].n + 1000 * r[i].k + 10000 * r[i].flag + r[i].tail;
  *out = s; return (int32_t)sizeof(rec_t);
}
int32_t fill3(double* a, int64_t d0, int64_t d1, int64_t d2) {    /* C order [d2][d1][d0] = a Julia Array{Float64}(undef, d0, d1, d2) */
  for (int64_t k = 0; k < d2; ++k) for (int64_t j = 0; j < d1; ++j) for (int64_t i = 0; i < d0; ++i) a[(k * d1 + j) * d0 + i] = 100 * k + 10 * j + i;
  return 0;
}
int32_t make_handle(void** out) { *out = (void*)0x5150; return 0; }
int64_t use_handle(void* h, int32_t* counter) { if (counter) *counter += 7; return (int64_t)(intptr_t)h; }
const char* last_message(void) { strcpy(msg, "from C"); return msg; }
uint64_t mask48(uint64_t x) { return x & 0xffffffffffffULL; }
void nothing(void) {}
"""


@pytest.fixture(scope="module")
def ffi_lib(tmp_path_factory):
    import subprocess
    d = tmp_path_factory.mktemp("ffi")
    src, so = d / "ffi_test.c", d / "libffi_test.so"
    src.write_text(FFI_C)
    subprocess.check_call(["gcc", "-O1", "-shared", "-fPIC", "-o", str(so), str(src)])
    return str(so)


def test_ccall_marshals_like_julia(ffi_lib):
    """struct arrays by field order with C alignment, column-major arrays, Ref out-parameters, Ptr{Cvoid} handles, Cstring,
    C_NULL, unsigned 64-bit values, Cvoid returns — against a real C library (gcc)."""
    it = Interp()
    it.genv.vars["LIB"] = ffi_lib
    out = it.run_string('''
struct Rec
  a::Cdouble; b::Float64; n::Int64; k::Int32; flag::Int32; tail::Cdouble
end
recs = [Rec(1.5, 2.0, 3, 4, true, 0.25), Rec(0.5, 1.0, 1, 1, false, 0.125)]
s = Ref{Cdouble}(0.0)
sz = ccall((:rec_sum, LIB), Int32, (Ptr{Rec}, Int64, Ptr{Cdouble}), recs, length(recs), s)
A = Array{Float64}(undef, 2, 3, 4)
rc = ccall((:fill3, LIB), Int32, (Ptr{Float64}, Int64, Int64, Int64), A, 2, 3, 4)
h = Ref{Ptr{Cvoid}}(C_NULL)
ccall((:make_handle, LIB), Int32, (Ptr{Ptr{Cvoid}},), h)
cnt = Ref{Int32}(5)
hv = ccall((:use_handle, LIB), Int64, (Ptr{Cvoid}, Ptr{Int32}), h[], cnt)
hv0 = ccall((:use_handle, LIB), Int64, (Ptr{Cvoid}, Ptr{Int32}), h[], C_NULL)
msg = unsafe_string(ccall((:last_message, LIB), Cstring, ()))
m = ccall((:mask48, LIB), UInt64, (UInt64,), UInt64(0x123456789abcdef0) & 0xffffffffffffffff)
nothing_back = ccall((:nothing, LIB), Cvoid, ())
(sz, s[], rc, A[2, 3, 4], A[1, 2, 3], A[:, 1, 2], hv, cnt[], hv0, msg, m, nothing_back)
''')
    sz, s, rc, a234, a123, col, hv, cnt, hv0, msg, m, nb = out
    assert sz == 40
    assert s == (1.5 + 20 + 300 + 4000 + 10000 + 0.25) + (0.5 + 10 + 100 + 1000 + 0 + 0.125)
    assert rc == 0 and a234 == 100 * 3 + 10 * 2 + 1 and a123 == 100 * 2 + 10 * 1 + 0
    assert list(col) == [100.0, 101.0]
    assert hv == 0x5150 and cnt == 12 and hv0 == 0x5150 and msg == "from C"
    assert m == 0x123456789abcdef0 & 0xffffffffffff and nb is None


def test_ccall_errors_are_loud(ffi_lib):
    it = Interp()
    it.genv.vars["LIB"] = ffi_lib
    with pytest.raises(JlError, match="could not load symbol"):
        it.run_string('ccall((:no_such_function, LIB), Int32, ())')
    with pytest.raises(JlError, match="declares 2 argument types but 1 arguments"):
        it.run_string('ccall((:use_handle, LIB), Int64, (Ptr{Cvoid}, Ptr{Int32}), C_NULL)')
    with pytest.raises(JlError, match="could not load library"):
        it.run_string('ccall((:f, "/nonexistent/lib.so"), Int32, ())')
    with pytest.raises(JlError, match="InexactError"):
        it.run_string('ccall((:fill3, LIB), Int32, (Ptr{Float64}, Int64, Int64, Int64), C_NULL, 1.5, 1, 1)')
    with pytest.raises(JlError, match="passed as Ptr"):
        it.run_string('ccall((:fill3, LIB), Int32, (Ptr{Float64}, Int64, Int64, Int64), [1, 2, 3], 3, 1, 1)')
