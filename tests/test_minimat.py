"""oracle/minimat -- the MATLAB-subset interpreter that executes the UNMODIFIED reference -- checked three ways.

1. Language semantics: known MATLAB behaviours (column-major linear indexing, ``end``, growth on assignment, implicit expansion,
   value semantics, white space inside brackets, transpose vs quote, ``nargin`` / ``nargout``, nested functions sharing the
   parent workspace, closures, classdef with inheritance and method dispatch, command syntax, ``fread`` / ``fwrite``).
2. Against numbers REAL MATLAB produced and the reference still holds (needs a checkout of it in ``SWRT_REFERENCE_DIR``):
   the unmodified ``qg_flow_ray_trace/qgsw_raytrace.m`` run under minimat prints the header lines MATLAB R2020b printed into
   the shipped SLURM logs, its ``pv_time`` stream lands within 2 ulps of the stored one, the unmodified ``rsw/k2g.m`` /
   ``fulspec.m`` reproduce the grid fields stored in ``rsw/matlab.mat``, and the unmodified solver ``rsw/swk.m`` run for 300
   steps from the initial condition in that file reproduces the whole workspace MATLAB dumped at step 300.
3. The committed hot-path goldens (``tests/golden/octave_out``) are what running the unmodified reference gives: a slice of
   the recipe is re-run here and compared bit for bit, and the sha256 of every executed reference file is checked.
"""
import io
import json
import os
import sys
import textwrap
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests" / "golden"))

from oracle.minimat import Interp, MatlabError, MStruct, MCell      # noqa: E402

# a checkout of the original MATLAB project (ndefilippis/SWRaytracing), which this repository does not carry
REF = Path(os.environ.get("SWRT_REFERENCE_DIR", "")).absolute()
HAVE_REF = bool(os.environ.get("SWRT_REFERENCE_DIR")) and (REF / "ode_symplectic.m").exists()
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="set SWRT_REFERENCE_DIR to a checkout of the original MATLAB project")
GOLD = ROOT / "tests" / "golden"


def run(src, **kw):
    buf = io.StringIO()
    I = Interp(out=buf, **kw)
    fr = I.run(textwrap.dedent(src))
    return fr.vars, buf.getvalue()


def arr(*rows):
    return np.array(rows, dtype=np.float64)


# ---------------------------------------------------------------------------------------------------- 1. semantics
def test_matrix_literals_and_white_space_rules():
    v, _ = run("""
        a = [1 2 3; 4 5 6];
        b = [1 -2];          % two elements
        c = [1 - 2];         % one
        d = [1 -2 + 3];      % 1 and 1
        e = [a(1,:) -1];
        f = [a', [7;8;9]];
        g = [1, 2
             3, 4];
        h = [a (1)];         % a and 1 side by side would not fit; MATLAB parses "a (1)" as two elements
    """.replace("h = [a (1)];", "h = [b (1)];"))
    assert np.array_equal(v["a"], arr([1, 2, 3], [4, 5, 6]))
    assert np.array_equal(v["b"], arr([1, -2]))
    assert v["c"] == -1.0
    assert np.array_equal(v["d"], arr([1, 1]))
    assert np.array_equal(v["e"], arr([1, 2, 3, -1]))
    assert np.array_equal(v["f"], arr([1, 4, 7], [2, 5, 8], [3, 6, 9]))
    assert np.array_equal(v["g"], arr([1, 2], [3, 4]))
    assert np.array_equal(v["h"], arr([1, -2, 1]))


def test_transpose_versus_quote():
    v, _ = run("""
        a = [1 2 3];
        b = a';
        c = a'*2;
        s = 'it''s';
        t = ['ab' 'cd'];
        u = {a', 'x'};
        w = [a' a'];
        z = (1+2i)';
        zz = (1+2i).';
    """)
    assert v["b"].shape == (3, 1) and v["c"].shape == (3, 1) and v["c"][2, 0] == 6
    assert v["s"] == "it's" and v["t"] == "abcd"
    assert v["u"].a[0, 0].shape == (3, 1) and v["u"].a[0, 1] == "x"
    assert v["w"].shape == (3, 2)
    assert v["z"] == complex(1, -2) and v["zz"] == complex(1, 2)


def test_indexing_is_column_major_one_based_with_end():
    v, _ = run("""
        a = [1 2 3; 4 5 6];
        l4 = a(4);                 % column-major: [1 4 2 5 3 6]
        col = a(:);
        last = a(end);
        e2 = a(end, end-1);
        r = a(2, :);
        m = a(:, [1 3]);
        lg = a(a > 2)';
        x3 = zeros(2, 3, 4); x3(2, 3, 4) = 7;
        f1 = x3(:, :, 4);
        f2 = x3(2, end);           % fewer subscripts than dimensions: the last one spans the rest (3*4 = 12)
        sz = size(x3(1, :, :));
        v1 = 10:-3:0;
        ev = v1(end:-1:1);
        rr = a(2, 2:end);
    """)
    assert v["l4"] == 5.0 and v["last"] == 6.0 and v["e2"] == 5.0
    assert np.array_equal(v["col"].ravel(), [1, 4, 2, 5, 3, 6]) and v["col"].shape == (6, 1)
    assert np.array_equal(v["r"], arr([4, 5, 6])) and np.array_equal(v["m"], arr([1, 3], [4, 6]))
    assert np.array_equal(v["lg"], arr([4, 5, 3, 6]))
    assert v["f1"][1, 2] == 7 and v["f2"] == 7.0
    assert np.array_equal(v["sz"], arr([1, 3, 4]))
    assert np.array_equal(v["v1"], arr([10, 7, 4, 1])) and np.array_equal(v["ev"], arr([1, 4, 7, 10]))
    assert np.array_equal(v["rr"], arr([5, 6]))


def test_assignment_grows_arrays_and_takes_extents_from_the_right_hand_side():
    v, _ = run("""
        w(3) = 1;                       % undefined -> 1x3 row
        c = zeros(2,1); c(4) = 9;       % a column stays a column
        U1(:,1) = [1;2;3];              % interpolate_U.m:5  (undefined, colon takes its extent from the right)
        U1(:,2) = [4;5;6];
        z = zeros(2,3); z(:,2) = [7;8];
        E = zeros(2,3); E(2,:) = [1;2;3];        % a column into a row slot: allowed, same number of elements
        x = zeros(3,2,4); x0 = ones(1,2,4); x(2,:,:) = x0;        % ode_symplectic.m:6
        f(1:2, 3:4) = [1 2; 3 4];       % read_field.m:86 on an undefined array
        q = 1:5; q([2 4]) = [];
        s = 'abc'; s(2) = 'X';
        g = zeros(2,2); g(:) = 1:4;
        b = zeros(2,2); b(3,3) = 1;
    """)
    assert np.array_equal(v["w"], arr([0, 0, 1])) and v["c"].shape == (4, 1) and v["c"][3, 0] == 9
    assert np.array_equal(v["U1"], arr([1, 4], [2, 5], [3, 6]))
    assert np.array_equal(v["z"], arr([0, 7, 0], [0, 8, 0])) and np.array_equal(v["E"], arr([0, 0, 0], [1, 2, 3]))
    assert v["x"].shape == (3, 2, 4) and v["x"][1].sum() == 8 and v["x"].sum() == 8
    assert np.array_equal(v["f"], arr([0, 0, 1, 2], [0, 0, 3, 4]))
    assert np.array_equal(v["q"], arr([1, 3, 5])) and v["s"] == "aXc"
    assert np.array_equal(v["g"], arr([1, 3], [2, 4])) and v["b"].shape == (3, 3)


def test_value_semantics_structs_cells_dynamic_fields():
    v, _ = run("""
        P.x = 1; P.k = 2;
        Q = P; Q.a = 5; Q.x = 9;               % make_octave_goldens.m:  Q = P; Q.a = 1
        s.a.b.c = 3;
        names = {'u', 'v'};
        bf.(names{2}) = 7;
        t = ['bf1_' names{1}];
        n = numel(names);
        c = cell(1, 2); c{2} = [1 2 3];
        a = [1 2 3]; b = a; b(2) = 0;
        isf = isfield(P, 'a');
    """)
    assert set(v["P"].f) == {"x", "k"} and v["P"].f["x"] == 1.0 and v["Q"].f["x"] == 9.0 and v["Q"].f["a"] == 5.0
    assert v["s"].f["a"].f["b"].f["c"] == 3.0 and v["bf"].f["v"] == 7.0 and v["t"] == "bf1_u" and v["n"] == 2.0
    assert np.array_equal(v["c"].a[0, 1], arr([1, 2, 3]))
    assert np.array_equal(v["a"], arr([1, 2, 3])) and np.array_equal(v["b"], arr([1, 0, 3])) and v["isf"] is False


def test_arithmetic_expansion_precedence_and_scalars():
    v, _ = run("""
        p1 = -2^2;  p2 = 2^-1;  p3 = 2^3^2;  p4 = -2^-2;
        r = [1;2;3] + [10 20];                  % implicit expansion 3x1 + 1x2
        k = ones(1,2,3); om = 2*ones(1,1,3); q = k ./ om;          % ode_symplectic.m:12  (1x2xN ./ 1x1xN)
        d = dot(k, k, 2);
        m = mod(-1, 5);  m2 = mod(5.5, 2);  m3 = mod(-1e-17, 32);  m0 = mod(3, 0);
        bump = 10^(-13);
        c = (1+2i)*(1-2i);                      % complex result with zero imaginary part is real
        cr = isreal(c);
        e = [1 2 3] == [1 5 3];
        t = ~isempty([]) | 1;
        z = 1/0;  nz = -1/0;
        ch = 5 < 7 <= 1;                         % (5<7) <= 1 -> true: the chained comparison of qgsw_raytrace.m:202
        i2 = 3 + 2*i;
        col = (1:3)';
        mm = [1 2; 3 4] * [1; 1];
        sq = sqrt(-4);
    """)
    assert v["p1"] == -4.0 and v["p2"] == 0.5 and v["p3"] == 64.0 and v["p4"] == -0.25
    assert np.array_equal(v["r"], arr([11, 21], [12, 22], [13, 23]))
    assert v["q"].shape == (1, 2, 3) and (v["q"] == 0.5).all() and v["d"].shape == (1, 1, 3) and (v["d"] == 2).all()
    assert v["m"] == 4.0 and v["m2"] == 1.5 and v["m3"] == 32.0 and v["m0"] == 3.0
    assert v["bump"] == 10.0 ** -13
    assert v["c"] == 5.0 and type(v["c"]) is float and v["cr"] is True
    assert np.array_equal(v["e"], np.array([[True, False, True]])) and v["t"] is True
    assert v["z"] == np.inf and v["nz"] == -np.inf and v["ch"] is True and v["i2"] == complex(3, 2)
    assert v["col"].shape == (3, 1) and np.array_equal(v["mm"], arr([3], [7])) and v["sq"] == 2j


def test_control_flow_switch_and_one_line_forms():
    v, out = run("""
        k = 0; for i = 1:3, k = k + i; end
        n = 0; while n < 10, n = n + 3; if n > 5, break, end, end
        x = 2;
        switch x
          case 1, r = 'one';
          case {2, 3}
            r = 'two-three';
          otherwise
            r = 'other';
        end
        switch 'abc', case 'abd', s = 1; case 'abc', s = 2; end
        cols = 0; for c = [1 2; 3 4], cols = cols + c(2); end
        status = 1;
        if status~=0 disp('bad'), end            % write_field.m:35: no comma after the condition
        if (1 > 2 & undefined_thing == 1), y = 1; else, y = 2; end     % '&' short-circuits in an if (read_field.m:40)
        fprintf('%d %f %s %5.2f%%\\n', 3, 2.5, 'hi', 12.345);
        fprintf("%d,", [1 2 3]); fprintf("\\n");
        fprintf('%d\\n', 2.5);
    """)
    assert v["k"] == 6.0 and v["n"] == 6.0 and v["r"] == "two-three" and v["s"] == 2.0 and v["cols"] == 7.0 and v["y"] == 2.0
    assert out == "bad\n3 2.500000 hi 12.35%\n1,2,3,\n2.500000e+00\n"


def test_functions_nargin_nargout_nested_closures(tmp_path):
    (tmp_path / "outer.m").write_text(textwrap.dedent("""
        function [a, b, c] = outer(x, y)
            if nargin < 2, y = 10; end
            a = x + y;
            if nargout > 1, b = helper(a); end
            if nargout > 2, c = 3; end
        end
        function r = helper(v)
            r = v * 2;
        end
    """))
    (tmp_path / "stepper.m").write_text(textwrap.dedent("""
        function [x, count] = stepper(x0, n, scale)
            count = 0;
            gain = @(v) (scale * v);             % anonymous function capturing a variable
            function y = bump(y0, dt)            % nested: shares 'count' and 'gain' with the parent, y0 / dt / y are its own
                y = y0 + dt * gain(1);
                count = count + 1;
            end
            x = x0;
            for i = 1:n
                x = apply_twice(x, @bump);
            end
        end
        function y = apply_twice(y0, f)
            y = f(f(y0, 0.5), 0.5);
        end
    """))
    (tmp_path / "noend.m").write_text("function r = noend(a)\nr = sub(a) + 1;\n\nfunction q = sub(a)\nq = 2*a;\n")
    (tmp_path / "logger.m").write_text(textwrap.dedent("""
        function h = logger(maxlevel)
            function log_func(fmt, level, varargin)
                if level <= maxlevel
                    fprintf(fmt, varargin{:});
                end
            end
            h = @log_func;
        end
    """))
    v, out = run("""
        a1 = outer(1);
        [a2, b2] = outer(1, 2);
        [~, ~, c3] = outer(1, 2);
        [x, cnt] = stepper(0, 3, 2);
        r = noend(5);
        lg = logger(1);
        lg("n=%d\\n", 1, 42);
        lg("hidden %d\\n", 2, 43);
    """, cwd=str(tmp_path))
    assert v["a1"] == 11.0 and v["a2"] == 3.0 and v["b2"] == 6.0 and v["c3"] == 3.0
    assert v["x"] == 6.0 and v["cnt"] == 6.0 and v["r"] == 11.0
    assert out == "n=42\n"
    with pytest.raises(MatlabError, match="not assigned|outputs requested"):
        run("[a, b, c] = outer(1);" .replace("outer(1)", "only_one(1)"), cwd=str(_one_output_dir(tmp_path)))


def _one_output_dir(tmp_path):
    (tmp_path / "only_one.m").write_text("function [a, b] = only_one(x)\na = x;\n")
    return tmp_path


def test_classdef_inheritance_and_method_dispatch(tmp_path):
    (tmp_path / "Base.m").write_text(textwrap.dedent("""
        classdef Base
            methods(Abstract)
                v = value(obj, x)
            end
            methods
                function r = twice(obj, x)
                    r = 2 * obj.value(x);
                end
            end
        end
    """))
    (tmp_path / "Derived.m").write_text(textwrap.dedent("""
        classdef Derived < Base
            properties
                gain, info, L
            end
            methods
                function obj = Derived(g)
                    addpath ./sub/
                    obj.gain = g;
                    obj.info.name = 'd';
                    obj.info.n = 3;
                end
                function v = value(obj, x, t)
                    v = obj.gain * x + from_sub();
                end
            end
        end
    """))
    (tmp_path / "sub").mkdir()
    (tmp_path / "sub" / "from_sub.m").write_text("function r = from_sub()\nr = 100;\n")
    v, _ = run("""
        d = Derived(3);
        a = d.value(2);
        b = d.twice(2);          % inherited method calling the subclass's through obj.value(...)
        c = twice(d, 1);         % function syntax dispatches on the object too
        g = d.gain; nm = d.info.name;
        e = d; e.gain = 0;       % value class: d is not changed
        a2 = d.value(2);
        cls = class(d); ok = isa(d, 'Base');
    """, cwd=str(tmp_path))
    assert v["a"] == 106.0 and v["b"] == 212.0 and v["c"] == 206.0 and v["g"] == 3.0 and v["nm"] == "d" and v["a2"] == 106.0
    assert v["cls"] == "Derived" and v["ok"] is True


def test_path_precedence_current_folder_then_addpath_order(tmp_path):
    for d, val in (("a", 1), ("b", 2)):
        (tmp_path / d).mkdir()
        (tmp_path / d / "which_one.m").write_text(f"function r = which_one()\nr = {val};\n")
    v, _ = run("""
        addpath('a'); addpath('b');        % addpath prepends: b wins
        r1 = which_one();
        addpath a                           % command syntax; moves a to the front
        r2 = which_one();
    """, cwd=str(tmp_path))
    assert v["r1"] == 2.0 and v["r2"] == 1.0


def test_binary_files_round_trip_like_write_field_and_read_field(tmp_path):
    v, _ = run(f"""
        A = [1 2 3; 4 5 6];
        fid = fopen('{tmp_path}/t.bin', 'a', 'n');
        fseek(fid, 0, -1);
        n = fwrite(fid, A, 'real*8');
        fclose(fid);
        [fid, msg] = fopen('{tmp_path}/t.bin', 'r', 'n');
        B = fread(fid, [2 inf], 'real*8');
        fclose(fid);
        [bad, why] = fopen('{tmp_path}/missing.bin', 'r');
    """)
    assert v["n"] == 6.0 and np.array_equal(v["B"], v["A"]) and v["bad"] == -1.0 and v["why"]
    assert np.array_equal(np.fromfile(tmp_path / "t.bin"), [1, 4, 2, 5, 3, 6])            # column-major on disk


def test_rand_is_matlabs_mersenne_twister_stream():
    """rng(s); rand(m,n) = mt19937ar 53-bit doubles filled column-major (the known MATLAB / numpy RandomState identity);
    first draws of rng(0) are MATLAB's documented 0.8147 0.9058 0.1270 0.9134 0.6324."""
    v, _ = run("rng(0); r = rand(1, 5); rng(146); p = rand(3, 2);")
    assert np.allclose(v["r"], [[0.8147, 0.9058, 0.1270, 0.9134, 0.6324]], atol=5e-5)
    ref = np.random.RandomState(146).random_sample(6)
    assert np.array_equal(v["p"], ref.reshape(3, 2, order="F"))


def test_fft_kit_conventions():
    v, _ = run("""
        x = [1 2 3 4; 5 6 7 8; 9 10 11 12; 13 14 15 17];
        X = fft2(x);
        y = ifft2(X);                  % conjugate-symmetric input -> real output, like MATLAB
        yr = isreal(y);
        s = fftshift([1 2 3 4 5]);  is_ = ifftshift([1 2 3 4 5]);
        [A, B] = ndgrid(-1:1, 0:1);
        [XX, YY] = meshgrid([1 2 3], [10 20]);
        ls = linspace(-1, 1, 5);
    """)
    assert v["yr"] is True and np.allclose(v["y"], v["x"], atol=1e-14)
    assert np.array_equal(v["s"], arr([4, 5, 1, 2, 3])) and np.array_equal(v["is_"], arr([3, 4, 5, 1, 2]))
    assert np.array_equal(v["A"], arr([-1, -1], [0, 0], [1, 1])) and np.array_equal(v["B"], arr([0, 1], [0, 1], [0, 1]))
    assert np.array_equal(v["XX"], arr([1, 2, 3], [1, 2, 3])) and np.array_equal(v["YY"], arr([10, 10, 10], [20, 20, 20]))
    assert np.array_equal(v["ls"], arr([-1, -0.5, 0, 0.5, 1]))


def test_errors_are_matlabs():
    for src, pat in (("a = [1 2 3]; a(4)", "out of bounds"), ("a = [1 2 3]; a(0)", "positive integer"),
                     ("x = undefined_name + 1;", "undefined function or variable"), ("a = [1 2; 3 4] + [1 2 3];", "incompatible"),
                     ("s.a = 1; s.b", "non-existent field"), ("error('boom %d', 3)", "boom 3"), ("assert(1 == 2)", "Assertion")):
        with pytest.raises(MatlabError, match=pat):
            run(src)


@needs_ref
def test_every_m_file_of_the_reference_parses():
    """all 97 .m files of the reference -- scripts, functions with and without ``end``, nested functions, classdefs, command
    syntax, name=value arguments, block comments -- go through the lexer and parser"""
    from oracle.minimat.parser import parse_source
    files = sorted(REF.rglob("*.m"))
    assert len(files) >= 90
    kinds = {"script": 0, "function": 0, "class": 0}
    for f in files:
        kinds[parse_source(f.read_text(errors="replace"), str(f)).kind] += 1
    assert kinds["class"] >= 3 and kinds["function"] >= 30 and kinds["script"] >= 20


# ------------------------------------------------------------------------------------------ 2. against real MATLAB output
class _Stop(Exception):
    pass


def _qgsw_interp(tmp, npackets_done=None):
    (tmp / "data").mkdir(exist_ok=True)
    buf = io.StringIO()
    I = Interp(cwd=str(tmp), out=buf)
    I.path.insert(0, str(REF / "qg_flow_ray_trace"))
    # qgsw_raytrace.m:63 calls grid_U with five arguments; the committed grid_U.m (grid_U.m:1,11) has since grown a sixth,
    # ``shear_strength``, that it adds to u -- the call as committed fails in MATLAB too ("not enough input arguments").  The
    # logs predate that argument, so the shim passes shear_strength = 0 to the UNMODIFIED grid_U.m (u + 0 is exact).
    ref_grid_U = I.load_unit(str(REF / "qg_flow_ray_trace" / "grid_U.m")).main
    I.overrides["grid_U"] = lambda I_, args, nargout, frame: I_.call_funcdef(ref_grid_U, list(args) + [0.0], nargout, frame)
    return I, buf


@needs_ref
def test_grid_U_as_committed_needs_its_sixth_argument(tmp_path):
    """the premise of the shim above: MATLAB semantics, reproduced -- an unset parameter is an undefined variable"""
    I = Interp(cwd=str(tmp_path), out=io.StringIO())
    I.path.insert(0, str(REF / "qg_flow_ray_trace"))
    with pytest.raises(MatlabError, match="undefined function or variable 'shear_strength'"):
        I.run("[kx_,ky_] = ndgrid(-3:3,0:3); K2 = kx_.^2+ky_.^2; f = grid_U(ones(7,4), 3, K2, kx_, ky_);")


@needs_ref
@pytest.mark.parametrize("U_g,w0,delay,log", [(0.2, 2, 1000, "analysis/job-37011720/run-1/run.log"),
                                              (0.4, 8, 1000, "analysis/job-37011720/run-12/run.log"),
                                              (0.5, 2, 1200, "run.log")])          # run.log: spin-up 400 = 1200 / f
def test_unmodified_qgsw_raytrace_prints_what_matlab_printed(U_g, w0, delay, log, tmp_path):
    """qgsw_raytrace(256, 50, w0, 6000, 1000, U_g, 3, 1) as runqgsw_raytrace.sbatch:31 launches it: every header line that
    depends on arithmetic (rng(146) -> rand -> initial_q with its always-true chained comparison -> g2k -> grid_U -> 6 x k2g
    -> max -> sqrt -> U0 -> Fr, dt) equals the line MATLAB R2020b wrote, character for character.  'Simulation time' is left
    out (the logged runs used an earlier definition of T: 2000 = T_days, not T_days/Fr^2), and so is 'Time step' for the logs of
    job 36976465 and run.log, which ran with CFL 0.1 (qgsw_raytrace.m:29 is 0.05 as committed)."""
    I, buf = _qgsw_interp(tmp_path)

    def stop_after_header(_):
        if "Simulation progress" in buf.getvalue():
            raise _Stop()
    I.on_output = stop_after_header
    with pytest.raises(_Stop):
        I.call("qgsw_raytrace", 256, 50, w0, 6000, delay, U_g, 3, 1, nargout=0)
    mine = buf.getvalue().splitlines()
    theirs = (REF / log).read_text(errors="replace").splitlines()
    start = next(i for i, ln in enumerate(theirs) if ln.startswith("Resolution:"))
    theirs = theirs[start:start + 13]
    assert len(mine) >= 13
    skip = {"Simulation time"} | ({"Time step"} if "37011720" not in log else set())
    compared = 0
    for a, b in zip(mine[:13], theirs):
        key = a.split(":")[0]
        assert key == b.split(":")[0]
        if key in skip:
            continue
        assert a == b, (a, b)
        compared += 1
    assert compared >= 11
    # the packet files the script wrote through the reference's own write_field.m
    px = np.fromfile(tmp_path / "data" / "packet_x.bin")
    pk = np.fromfile(tmp_path / "data" / "packet_k.bin")
    assert px.size == 100 and pk.size == 100 and np.all(np.abs(px) <= np.pi)
    assert np.allclose(np.hypot(pk[:50], pk[50:]), np.sqrt((w0 ** 2 - 1) * 9.0), rtol=1e-15)


@needs_ref
def test_unmodified_qgsw_raytrace_time_stream_matches_the_stored_one(tmp_path):
    """150 steps of the unmodified QG solver loop (update -> 4 x k2g + g2k per step, AB3, filter) with no packets: the frames
    ``write_field(t, pv_time_filename, frame)`` appends equal the stream the reference's own run stored
    (tests/golden/reference_runlogs.json <- qg_flow_ray_trace/data/.nfs...24, U_g = 0.2) to 2 ulps -- i.e. dt, hence U0, is
    MATLAB's to about one ulp (what is left is FFTW vs pocketfft round-off in the six k2g of grid_U)."""
    stored = np.array([float.fromhex(h) for h in json.loads((GOLD / "reference_runlogs.json").read_text())["pv_time"]["hex"][:4]])
    I, buf = _qgsw_interp(tmp_path)
    tfile = tmp_path / "data" / "pv_time.bin"

    def stop_after_frames(_):
        if tfile.exists() and tfile.stat().st_size >= 8 * 4:
            raise _Stop()
    I.on_output = stop_after_frames
    with pytest.raises(_Stop):
        I.call("qgsw_raytrace", 256, 0, 2, 6000, 1000, 0.2, 3, 1, nargout=0)
    I.close_all()
    t = np.fromfile(tfile)[:4]
    assert t[0] == 0.0 and np.all(np.abs(t - stored) <= 2 * np.spacing(stored)), (t, stored)
    # the PV frames themselves are not compared: ``update`` as committed adds ``r_drag * K2`` as a constant forcing
    # (qgsw_raytrace.m:285) and the field overflows within ~40 steps -- in MATLAB as here (oracle.qg_update restates the same
    # line); frame 1 is the initial condition the log header was computed from
    q0 = np.fromfile(tmp_path / "data" / "pv.bin")[:256 * 256]
    assert q0.size == 256 * 256 and np.isfinite(q0).all() and np.abs(q0).max() > 1.0


@needs_ref
def test_unmodified_k2g_reproduces_the_fields_in_matlabs_workspace_dump(tmp_path):
    """rsw/k2g.m + rsw/fulspec.m, unmodified, on the spectral state of rsw/matlab.mat (tests/golden/rsw_workspace_frame.npz):
    the rows of u, v, h, zeta MATLAB itself computed one line before the ``save`` (rsw/swk.m:205-213), to round-off."""
    R = np.load(GOLD / "rsw_workspace_frame.npz")
    I = Interp(cwd=str(tmp_path), out=io.StringIO())
    I.path.insert(0, str(REF / "rsw"))
    Sk, dm = R["Sk"], R["damask"].astype(np.float64)
    stride = int(R["row_stride"])
    fr = I.run("kmax = size(S1, 1)/2 - 0.5; [ikx_, iky_] = ndgrid(-kmax:kmax, 0:kmax); ikx_ = 1i*ikx_; iky_ = 1i*iky_;"
               "u = k2g(dm.*S1); v = k2g(dm.*S2); h = k2g(dm.*S3); zeta = k2g(dm.*(ikx_.*S2 - iky_.*S1)); ru = isreal(u);",
               frame=_frame_with(S1=Sk[:, :, 0], S2=Sk[:, :, 1], S3=Sk[:, :, 2], dm=dm))
    assert fr.vars["ru"] is True
    for name in ("u", "v", "h", "zeta"):
        rows = R[name + "_rows"]
        assert np.abs(rows).max() > 1e-2
        assert np.abs(fr.vars[name][::stride] - rows).max() <= 1e-15, name


@needs_ref
def test_unmodified_swk_run_for_300_steps_reproduces_matlabs_workspace(tmp_path):
    """The strongest pin of the interpreter.  ``rsw/matlab.mat`` is the workspace MATLAB dumped (the bare ``save`` of
    rsw/swk.m:178) at step n = 300 of ``swk(Sin, f, Cg, 10000, 100)`` -- and it still holds the inputs.  The unmodified
    ``rsw/swk.m`` (a 359-line pseudo-spectral rotating-shallow-water solver: globals, eight local functions closed by ``return``,
    Orszag-dealiased products through half-cell-shifted grids, AB3 with trapezoidal hyperviscosity, adaptive dt) is run by
    minimat from the same ``Sin`` for the same 300 steps and stopped at the same ``save``: the clock, time step, viscosity, Umax
    and counters MATLAB held are reproduced EXACTLY, the spectral state to 1e-15, the three saved right-hand sides to 1e-14 and
    the energy series to 1e-13 (the residue is FFTW vs pocketfft round-off through 300 nonlinear steps)."""
    sio = pytest.importorskip("scipy.io")
    names = ["Sin", "f", "Cg", "numsteps", "savestep", "n", "frame", "t", "dt", "nu", "Umax", "Sk", "Rk", "Rkm1", "Rkm2", "time", "ke", "pe"]
    M = sio.loadmat(str(REF / "rsw" / "matlab.mat"), variable_names=names)
    sc = lambda k: float(M[k][0, 0])
    assert sc("n") == 300 and sc("frame") == 4 and sc("savestep") == 100
    I = Interp(cwd=str(tmp_path), out=io.StringIO())
    I.path.insert(0, str(REF / "rsw"))
    snap = {}

    def save(I_, args, nargout, frame):                      # the bare ``save``: snapshot the workspace at n = 300 and stop there
        if I_.getvar(frame, "n") == sc("n"):
            for k in ("Sk", "Rk", "Rkm1", "Rkm2", "time", "ke", "pe", "dt", "nu", "Umax", "t", "frame", "n"):
                snap[k] = I_.getvar(frame, k)
            raise _Stop()
    I.overrides["save"] = save
    with pytest.raises(_Stop):
        I.call("swk", M["Sin"], sc("f"), sc("Cg"), sc("numsteps"), sc("savestep"), nargout=4)
    for k in ("t", "dt", "nu", "Umax", "frame", "n"):
        assert snap[k] == sc(k), (k, snap[k], sc(k))
    rel = lambda a, b: float(np.abs(np.asarray(a) - b).max() / np.abs(b).max())
    assert rel(snap["Sk"], M["Sk"]) < 1e-15
    for k in ("Rk", "Rkm1", "Rkm2"):
        assert rel(snap[k], M[k]) < 1e-14, k
    fr = int(sc("frame"))
    assert np.array_equal(np.asarray(snap["time"]).ravel()[:fr], M["time"].ravel()[:fr])
    for k in ("ke", "pe"):
        assert rel(np.asarray(snap[k]).ravel()[:fr], M[k].ravel()[:fr]) < 1e-13, k
    assert "Wrote frame >4 out of >100" in I.out.getvalue()


def _frame_with(**kw):
    from oracle.minimat import Frame, from_py
    fr = Frame(None)
    for k, v in kw.items():
        fr.vars[k] = from_py(np.asfortranarray(v))
    return fr


# ------------------------------------------------------------------------- 3. the committed goldens are the reference's output
EXPECTED = ("eval_lagrange", "eval_lagrange_qg", "interpU_lagrange", "rhs_lagrange", "scheme_eval", "scheme_gradU_times_k", "scheme_fields",
            "leapfrog100_scheme", "leapfrog20_scheme", "leapfrog_t", "cg_sw_fields", "rk4x3_packet_lagrange", "rk4x3_xka_lagrange")


def test_committed_goldens_are_complete_and_carry_their_provenance():
    out = GOLD / "octave_out"
    prov = json.loads((out / "PROVENANCE.json").read_text())
    assert prov["packets"] == "all" and "minimat" in prov["executor"]
    import hashlib
    for name in EXPECTED:
        f = out / f"{name}.bin"
        assert f.exists(), name
        assert hashlib.sha256(f.read_bytes()).hexdigest() == prov["outputs"][f.name]
    executed = set(prov["reference_files_executed"])
    assert {"ray_trace_sw/interpolate.m", "qg_flow_ray_trace/interpolate.m", "qg_flow_ray_trace/interpolate_U.m", "SpectralScheme.m", "RaytracingScheme.m",
            "ode_symplectic.m", "ray_trace_sw/cg_sw.m", "ray_trace_sw/step_packet.m", "ray_trace_sw/step_packet_xka.m",
            "qg_flow_ray_trace/read_field.m", "qg_flow_ray_trace/write_field.m"} <= executed
    assert {"rsw/g2k.m", "rsw/k2g.m", "rsw/fulspec.m"} <= executed       # SpectralScheme.m:8 puts ./rsw/ in front of the path


@needs_ref
def test_reference_files_are_the_ones_the_goldens_were_made_from():
    import hashlib
    prov = json.loads((GOLD / "octave_out" / "PROVENANCE.json").read_text())
    for rel, sha in prov["reference_files_executed"].items():
        assert hashlib.sha256((REF / rel).read_bytes()).hexdigest() == sha, rel


@needs_ref
def test_rerunning_a_slice_of_the_recipe_reproduces_the_committed_goldens(tmp_path):
    """make_octave_goldens.m on the first two packets, executed again here from the unmodified reference: every output equals
    the corresponding slice of the committed files bit for bit (packets are independent; the grid outputs do not depend on them)"""
    import run_reference_recipe as RR
    n = 2
    ind = RR.truncated_inputs(GOLD / "octave_in", n, tmp_path / "in")
    RR.run(REF, ind, tmp_path / "out", quiet=True)
    full_n = int(np.fromfile(GOLD / "octave_in" / "params.bin")[7])
    for name in EXPECTED:
        got = np.fromfile(tmp_path / "out" / f"{name}.bin")
        ref = np.fromfile(GOLD / "octave_out" / f"{name}.bin")
        if name in ("scheme_fields", "leapfrog_t"):
            assert np.array_equal(got, ref), name
        elif name == "cg_sw_fields":
            assert np.array_equal(got, ref), name                 # depends on packet 1 only
        else:
            rows = ref.size // full_n
            assert np.array_equal(got.reshape(rows, n, order="F"), ref.reshape(rows, full_n, order="F")[:, :n]), name
