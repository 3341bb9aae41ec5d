"""The MATLAB-subset interpreter (oracle/mlab) that executes the reference's own functions/*.m to pin parity.

Two tiers, both CPU: language semantics on small snippets whose MATLAB results are known by definition of the
language, and - where KR_REFERENCE_DIR names a checkout of the reference - the reference's
unmodified sources executed live: every file parses, the committed golden file is reproduced bit for bit, and the
L1 recurrences agree with the oracle on fresh random inputs."""
import io
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import GOLDEN, ROOT, load_graph

from oracle.mlab import Interpreter, MatlabError, Cell, Struct

REFDIR = os.environ.get("KR_REFERENCE_DIR", "")
has_ref = pytest.mark.skipif(not (REFDIR and os.path.isdir(os.path.join(REFDIR, "functions"))),
                             reason="KR_REFERENCE_DIR names no checkout of the reference: the committed goldens stand in")


def run(src, tmp_path, **ws):
    p = tmp_path / "snippet.m"
    p.write_text(textwrap.dedent(src))
    I = Interpreter(path=[str(tmp_path)], stdout=io.StringIO())
    out = I.run_script(str(p), ws)
    return out, I


def val(x):
    return np.asarray(x).tolist()


def test_indexing_end_growth_and_value_semantics(tmp_path):
    ws, _ = run("""
        a = [1 2 3; 4 5 6];
        b = a;  b(2, 3) = 60;            % value semantics: a is untouched
        c = a(end, end);  d = a(:, end - 1)';  e = a(:)';  f = a(end);
        H = zeros(2, 0);  H(size(H, 1) + 2, size(H, 2) + 2) = 0;     % lanczos_krylov.m:84
        H(max(1, end - 3):end - 2, end - 1:end) = [1 2; 3 4];
        v = [];  v(3) = 7;               % growth of an empty along a row
        w = (1:5)';  w(7) = 1;           % growth of a column stays a column
        m = a(a > 2)';                   % logical mask: column-major order
        r = a(2, [true false true]);
        k = a([1 2; 2 1]);               % matrix subscript: the result has the subscript's shape
        z = 5:-1:1;  z([1 end]) = [];    % deletion
        s = a;  s(:, 2) = [];
    """, tmp_path)
    assert val(ws["a"]) == [[1, 2, 3], [4, 5, 6]] and val(ws["b"])[1][2] == 60
    assert val(ws["c"]) == [[6]] and val(ws["d"]) == [[2, 5]] and val(ws["e"]) == [[1, 4, 2, 5, 3, 6]] and val(ws["f"]) == [[6]]
    assert ws["H"].shape == (4, 2) and val(ws["H"]) == [[1, 2], [3, 4], [0, 0], [0, 0]]
    assert val(ws["v"]) == [[0, 0, 7]] and ws["w"].shape == (7, 1)
    assert val(ws["m"]) == [[4, 5, 3, 6]] and val(ws["r"]) == [[4, 6]] and val(ws["k"]) == [[1, 4], [4, 1]]
    assert val(ws["z"]) == [[4, 3, 2]] and val(ws["s"]) == [[1, 3], [4, 6]]


def test_matrix_literal_white_space_and_quotes(tmp_path):
    ws, _ = run("""
        a = 2;  b = 3;
        x = [a -b];  y = [a - b];  z = [a -b + 1];  t = [a' b'];  q = [0 -inf];
        u = [a, -b; b a];
        s = ['ab' 'c''d'];  n = [1, 2
             3, 4];
        e = 1./[2 4];  p = 2^-1;  g = -2^2;  h = [1 2]';
        l = {a, 'x'; [1 2], {}};
    """, tmp_path)
    assert val(ws["x"]) == [[2, -3]] and val(ws["y"]) == [[-1]] and val(ws["z"]) == [[2, -2]] and val(ws["t"]) == [[2, 3]]
    assert val(ws["q"]) == [[0, -np.inf]] and val(ws["u"]) == [[2, -3], [3, 2]] and ws["s"] == "abc'd"
    assert val(ws["n"]) == [[1, 2], [3, 4]] and val(ws["e"]) == [[0.5, 0.25]] and val(ws["p"]) == [[0.5]] and val(ws["g"]) == [[-4]]
    assert ws["h"].shape == (2, 1) and ws["l"].shape == (2, 2) and isinstance(ws["l"].a[1, 1], Cell)


def test_cells_comma_lists_and_nested_lvalues(tmp_path):
    ws, _ = run("""
        X = {{}};
        for h = 1:2, X = {X{:}, {}}; end       % function_multiple_entries.m:64-67
        X{2}{1} = [1 2];
        X{2}{2} = 5;
        X{2}{1}(3, 3) = 9;                      % function_multiple_entries.m:123
        Y = [{X{2}{2:2}}, [7 8]];               % cell ++ matrix wraps the matrix (fun_update.m:117)
        S = {};  S = [S, 4];  S = [S, 5];       % fun_update.m:104
        G{3} = 1;                               % brace assignment creates the cell
        n = numel(X);  c = {X{2}{:}};
    """, tmp_path)
    assert ws["X"].shape == (1, 3) and ws["X"].a[0, 1].shape == (1, 2)
    assert val(ws["X"].a[0, 1].a[0, 0]) == [[1, 2, 0], [0, 0, 0], [0, 0, 9]]
    assert ws["Y"].shape == (1, 2) and val(ws["Y"].a[0, 1]) == [[7, 8]]
    assert ws["S"].shape == (1, 2) and ws["G"].shape == (1, 3) and val(ws["n"]) == [[3]] and ws["c"].shape == (1, 2)


def test_functions_nargin_nargout_varargin_closures(tmp_path):
    (tmp_path / "two.m").write_text(textwrap.dedent("""
        function [a, b, c] = two(varargin)
        if nargin ~= 2 && nargin ~= 3
            error('Called with the wrong number of arguments');
        end
        a = nargin;  b = nargout;
        if nargout > 2, c = sub(varargin{:}); end
        end
        function s = sub(x, y, z)
        if ~exist('z', 'var'), z = 100; end
        s = x + y + z;
        end
    """))
    (tmp_path / "nest.m").write_text(textwrap.dedent("""
        function c = nest(A, m)
        n = 3;
        h = @inner;
        c = h('go', 2);
            function Z = inner(flag, X)
                if isequal(flag, 'go'), for i = 1:m, X = A * X; end, end
                Z = X + n;
            end
        end
    """))
    ws, I = run("""
        [p, q] = two(1, 2);
        [p3, q3, r3] = two(1, 2, 3);
        [~, onlyq] = two(1, 2);
        k = 10;  f = @(x) x + k;  k = 20;  fv = f(1);          % capture by value
        Af = 2;  Af = @(x) Af * x;  Af = @(x) Af(Af(x));  av = Af(1);   % mc_trace.m:33,49 style re-binding
        nv = nest(2, 3);
        msg = '';
        try
            two(1);
        catch err
            msg = err.message;
        end
        g = @exp;  same = isequal(g, @exp);  other = isequal(g, @sinh);  gv = g(0);
    """, tmp_path)
    assert val(ws["p"]) == [[2]] and val(ws["q"]) == [[2]] and val(ws["r3"]) == [[6]] and val(ws["onlyq"]) == [[2]]
    assert val(ws["fv"]) == [[11]] and val(ws["av"]) == [[4]] and val(ws["nv"]) == [[19]]
    assert ws["msg"].startswith("Called with the wrong number of arguments")
    assert val(ws["same"]) == [[True]] and val(ws["other"]) == [[False]] and val(ws["gv"]) == [[1]]


def test_control_flow_sparse_and_builtins(tmp_path):
    ws, _ = run("""
        A = sparse([1 2 2 3], [2 1 3 2], 1, 3, 3);
        sym = issymmetric(A);  nz = nnz(A);
        A(1, 2) = 0;  A(2, 1) = 0;  nz2 = nnz(A);          % krylov_miobi.m:128-129: entries set to 0 are dropped
        [i, j] = find(tril(A, -1));
        B = A + 1;  cls = issparse(B);  C = A * ones(3, 2);  D = 2 * A;  sp2 = issparse(D);
        c = [3 1 2 3];  [s, ix] = sort(c, 'descend');       % stable: the two 3s keep their order
        [mx, im] = max(c);  [mn, in] = min([4 2 2]);
        u = unique([3 1 3 2], 'stable');  d = setdiff([5 3 1], 3);
        t = 0;
        for col = [1 2; 3 4], t = t + col(2); end           % a for loop runs over COLUMNS
        w = 0;  while w < 3, w = w + 1; if w == 2, continue, end, end
        switch 'min'
            case 'mult', o = 1;
            case {'min', 'max'}, o = 2;
            otherwise, o = 3;
        end
        e = isempty([]) && ~isempty(0);  sc = 1:0;  ne = numel(sc);
        if [1 1 0], allt = 1; else, allt = 0; end          % an array condition is true only if ALL are nonzero
        x = [1 2; 3 4] \\ [5; 6];  y = [5 6] / [1 2; 3 4];
        n2 = norm([3 4]);  ni = norm([1 -2; 3 4], inf);  n1 = norm([1 -2; 3 4], 1);  nf = norm([3 4], 'fro');
        st = sprintf('%d,%.2f,%s', 3, 2.5, 'ok');
    """, tmp_path)
    assert val(ws["sym"]) == [[True]] and val(ws["nz"]) == [[4]] and val(ws["nz2"]) == [[2]]
    assert val(ws["i"]) == [[3]] and val(ws["j"]) == [[2]] and val(ws["cls"]) == [[False]] and val(ws["sp2"]) == [[True]]
    assert val(ws["C"]) == [[0, 0], [1, 1], [1, 1]]
    assert val(ws["s"]) == [[3, 3, 2, 1]] and val(ws["ix"]) == [[1, 4, 3, 2]]
    assert val(ws["im"]) == [[1]] and val(ws["in"]) == [[2]] and val(ws["u"]) == [[3, 1, 2]] and val(ws["d"]) == [[1, 5]]
    assert val(ws["t"]) == [[7]] and val(ws["o"]) == [[2]] and val(ws["e"]) == [[True]] and val(ws["ne"]) == [[0]] and val(ws["allt"]) == [[0]]
    assert np.allclose(ws["x"], [[-4], [4.5]]) and np.allclose(ws["y"], [[-1, 2]])
    assert val(ws["n2"]) == [[5]] and val(ws["ni"]) == [[7]] and val(ws["n1"]) == [[6]] and val(ws["nf"]) == [[5]]
    assert ws["st"] == "3,2.50,ok"


def test_idioms_of_the_reference_sources(tmp_path):
    """The exact statements the reference leans on, each with the value MATLAB's semantics prescribe."""
    # comments name the reference lines each idiom comes from: for-range evaluated once (function_multiple_entries.m:
    # 110,146), row deletion by index list (krylov_miobi.m:126), implicit expansion (greedy_krylov.m:66), lag buffer
    # (trace_fun_update.m:117), `C (C == 0) = inf` and blank-separated outputs (expmv.m:63-66), sparse hash table
    # (fun_and_grad_krylov_exp.m:52-53), stable descending sort + first match (find_top_edges.m:25-31), row() lookup
    # (function_multiple_entries.m:45), edge2low_rank.m:6-12, `if` on a size vector (function_multiple_entries.m:122),
    # matrix-to-handle rebinding (mc_trace.m:32-34)
    ws, _ = run("""
        notconv = [1 2 3 4];  seen = [];
        for h = notconv
            notconv = setdiff(notconv, h);
            seen = [seen h];
        end
        E = [1 2; 3 4; 5 6; 7 8];  k = 2;
        E2 = E([1:k-1, k+1:end], :);
        tmp = [5 6];  ind = find(prod(E == tmp, 2));
        Xstop = [1 2];  Xm = 3;  d = 2;  Xstop = [Xstop(2:d), Xm];
        C = [0 3; 2 0; 5 1];  C (C == 0) = inf;  [cost, m] = min(min(C));
        [cst m2] = min([4; 2; 2]);
        aux = [3; 7; 9];  iaux = sparse(max(aux), 1);  iaux(aux) = [1:3]';  i7 = full(iaux(7));
        c = [0.5 0.9 0.5 0.9 0.1];  [~, order] = sort(c, 'descend');
        sc = sort(c, 'descend');  first = find(sc == c(3), 1);
        I = unique([4; 2; 4; 9; 2], 'stable')';  row = @(t) sum((I == t) .* [1:length(I)]);  r9 = row(9);
        t1 = [2; 2; 5];  t2 = [5; 7; 7];  ut = unique([t1; t2]);
        U = sparse(ut, 1:length(ut), 1, 8, length(ut));  B = zeros(length(ut));
        for j = 1:length(t1)
            a = find(t1(j) == ut);  b = find(t2(j) == ut);  B(a, b) = -1;  B(b, a) = -1;
        end
        S = full(U * B * U');
        H = reshape(1:16, 4, 4);  H(1:end-2, end-1:end) = H(1:end-2, end-1:end) + [1 1; 1 1];
        nn = 3;  X = [1 2; 3 4];  if nn > size(X), X(nn, nn) = 0; end
        Afun = [2 0; 0 3];  if isfloat(Afun), Afun = @(x) Afun * x; end
        v = Afun([1; 1]);
        n17 = sprintf('%.17g', 0.1);
    """, tmp_path)
    assert val(ws["seen"]) == [[1, 2, 3, 4]] and ws["notconv"].size == 0
    assert val(ws["E2"]) == [[1, 2], [5, 6], [7, 8]] and val(ws["ind"]) == [[3]] and val(ws["Xstop"]) == [[2, 3]]
    assert val(ws["cost"]) == [[1]] and val(ws["m"]) == [[2]] and val(ws["cst"]) == [[2]] and val(ws["m2"]) == [[2]]
    assert val(ws["i7"]) == [[2]] and val(ws["order"]) == [[2, 4, 1, 3, 5]] and val(ws["first"]) == [[3]] and val(ws["r9"]) == [[3]]
    S = np.zeros((8, 8))
    for a, b in ((2, 5), (2, 7), (5, 7)):
        S[a - 1, b - 1] = S[b - 1, a - 1] = -1
    assert np.array_equal(ws["S"], S)
    assert val(ws["H"])[0][2:] == [10, 14] and val(ws["H"])[1][2:] == [11, 15] and val(ws["H"])[2][2:] == [11, 15]
    assert ws["X"].shape == (3, 3) and val(ws["v"]) == [[2], [3]] and ws["n17"] == "0.10000000000000001"


def test_errors_carry_file_and_line(tmp_path):
    with pytest.raises(MatlabError) as e:
        run("a = [1 2 3];\nb = a(4);\n", tmp_path)
    assert "Index exceeds" in str(e.value) and "snippet.m:2" in str(e.value)


# ----------------------------------------------------------------------------------------- the reference itself, live
@has_ref
def test_every_reference_function_file_parses():
    import glob
    from oracle.mlab.parser import parse_source
    files = sorted(glob.glob(os.path.join(REFDIR, "functions", "*.m")))
    assert len(files) == 22
    for f in files:
        body, funs = parse_source(open(f, errors="replace").read(), f)
        assert funs and funs[0].name == os.path.splitext(os.path.basename(f))[0].replace("arnoldi_krylov", "poly_krylov")


@has_ref
def test_committed_goldens_are_what_the_reference_sources_produce():
    """Re-runs scripts/make_reference_goldens.m over the reference's functions/*.m: bit-for-bit the committed file."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "run_reference_goldens.py"), "--refdir", REFDIR,
                        "--check"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "reproduced bit for bit" in r.stdout
    prov = json.load(open(os.path.join(GOLDEN, "reference_golden.provenance.json")))
    import hashlib
    for rel, h in prov["reference_files_executed"].items():
        assert hashlib.sha256(open(os.path.join(REFDIR, rel), "rb").read()).hexdigest() == h, rel


@has_ref
def test_reference_krylov_recurrences_live_against_the_oracle():
    """lanczos_krylov.m / arnoldi_krylov.m executed from source on fresh random blocks: V, H (K) of the oracle are
    the SAME matrices (the same LAPACK calls in the same order), not merely equivalent bases."""
    import oracle as O
    I = Interpreter(path=[os.path.join(REFDIR, "functions")], stdout=io.StringIO())
    A = sp.csc_matrix(load_graph("oregon_A1")).astype(np.float64)
    rng = np.random.default_rng(7)
    for bs in (1, 2, 5):
        b = rng.standard_normal((A.shape[0], bs))
        V, H, p, lk = I.call("lanczos_krylov", A, b, nargout=4)
        V2, H2, p2, lk2 = O.lanczos_krylov(A, b)
        for _ in range(3):
            V, H, p, lk = I.call("lanczos_krylov", V, H, p, nargout=4)
            V2, H2, p2, lk2 = O.lanczos_krylov(V2, H2, p2)
        assert np.max(np.abs(V - V2)) <= 1e-13 and np.max(np.abs(H - H2)) <= 1e-12 * np.max(np.abs(H))
        V, K, H, p, lk = I.call("arnoldi_krylov", A, b, nargout=5)
        V2, K2, H2, p2, lk2 = O.arnoldi_krylov(A, b)
        for _ in range(3):
            V, K, H, p, lk = I.call("arnoldi_krylov", V, K, H, p, nargout=5)
            V2, K2, H2, p2, lk2 = O.arnoldi_krylov(V2, K2, H2, p2)
        assert np.max(np.abs(V - V2)) <= 1e-13 and np.array_equal(K, K2) and np.max(np.abs(H - H2)) <= 1e-12 * np.max(np.abs(H))


@has_ref
def test_reference_error_strings_live():
    """The error() texts of the reference, raised by the reference's own lines."""
    I = Interpreter(path=[os.path.join(REFDIR, "functions")], stdout=io.StringIO())
    A = sp.csc_matrix(load_graph("oregon_A0")).astype(np.float64)
    with pytest.raises(MatlabError, match="Called with the wrong number of arguments"):
        I.call("lanczos_krylov", A, nargout=2)
    with pytest.raises(MatlabError, match="The block vector b has wrong number of rows"):
        I.call("lanczos_krylov", A, np.ones((3, 1)), nargout=2)
    with pytest.raises(MatlabError, match="The matrix A should be square"):
        I.call("lanczos_krylov", A[:, :10], np.ones((A.shape[0], 1)), nargout=2)
    Au = A.copy().tolil()
    Au[0, 5] = 3.0
    with pytest.raises(MatlabError, match="KRYLOV_MIOBI:: Adjacency matrix should be symmetric"):
        I.call("krylov_miobi", sp.csc_matrix(Au), 1, nargout=1)
    with pytest.raises(MatlabError, match="Invalid p_max or m_max"):
        I.call("select_taylor_degree", A, np.ones((A.shape[0], 1)), 70, 8, "double", False, False, nargout=1)
    with pytest.raises(MatlabError, match="Unsupported rational Krylov yet"):
        I.call("function_multiple_entries", A, np.array([[1.0, 2.0]]), I.call("str2func", "exp")[0], 1e-8, 10,
               np.array([[1.0, 2.0]]), 0, nargout=1)
