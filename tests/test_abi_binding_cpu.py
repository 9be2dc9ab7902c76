"""CPU checks of the ctypes binding that _native.py builds from include/pn12_b200.h: every declared function gets the
header's parameter count and return type, a few signatures element by element, the structs gcc's layout, and the parser
refuses what it does not understand instead of binding it with ctypes' default int conversion."""
import ctypes as C
import re

import pytest

from pointnet12_b200 import _native as nv

vp, i64, i32, f32 = C.c_void_p, C.c_int64, C.c_int, C.c_float


def test_every_declared_function_is_bound_with_the_headers_arity_and_return_type():
    # a separate, deliberately plain read of the prototypes: the header's prototypes have no parentheses in their parameters
    text = re.sub(r"/\*.*?\*/", "", open(nv.HEADER).read(), flags=re.S)
    protos = re.findall(r"(int|size_t|const char\*)\s+(pn_\w+)\(([^)]*)\);", text)
    assert sorted(name for _, name, _ in protos) == nv.declared_symbols()
    lib = nv.lib()
    returns = {"int": C.c_int, "size_t": C.c_size_t, "const char*": C.c_char_p}
    for ret, name, params in protos:
        fn = getattr(lib, name)
        n = 0 if params.strip() == "void" else params.count(",") + 1
        assert len(fn.argtypes) == n, name
        assert fn.restype is returns[ret], name


@pytest.mark.parametrize("name,argtypes,restype", [
    ("pn_fps_f32", [vp, i64, i64, i64, i32, i32, i32, vp, vp, vp, vp], C.c_int),
    ("pn_fp_mlp_bf16x3", [vp, vp, vp, i64, i64, i64, i32, vp, i64, i64, i64, i32, i32, vp, vp, i32, vp, i64, i64, vp, i64,
                          i32, i32, i32, vp, i64, vp, vp], C.c_int),
    ("pn_train_gemm_bf16x3", [vp, i64, i64, i32, vp, vp, i32, vp, i32, vp, i32, vp, i64, vp, vp, vp, vp], C.c_int),
    ("pn_three_interpolate_bwd_xyz_det_f32", [vp, i64, i32, i32, vp, vp, vp, i64, i64, i64, vp, i64, i64, i64, vp, i64, i64,
                                              i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp], C.c_int),
    ("pn_adam_f32", [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i64, f32, vp], C.c_int),
    ("pn_scan_workspace_bytes", [i32, i64], C.c_size_t),
    ("pn_last_error_string", [], C.c_char_p),
    ("pn_mlp_resident_groups", [vp], C.c_int),
])
def test_pinned_signatures(name, argtypes, restype):
    fn = getattr(nv.lib(), name)
    assert list(fn.argtypes) == argtypes
    assert fn.restype is restype


@pytest.mark.parametrize("struct,size,offsets", [
    (nv.LaunchOpts, 40, {"mlp_passes": 0, "fps_exchange": 20, "tile_counter": 24, "mlp_debug": 32}),
    (nv.MlpDesc, 76, {"nlayers": 0, "cin": 4, "cout": 28, "relu": 52}),
    (nv.TrainPackItem, 32, {"w": 0, "out": 8, "cin": 16, "cout": 20, "transposed": 24, "reserved": 28}),
])
def test_struct_layouts_match_gcc(struct, size, offsets):
    assert C.sizeof(struct) == size
    assert {f: getattr(struct, f).offset for f in offsets} == offsets
    assert nv.MLP_MAX_LAYERS == 6 and nv.MlpDesc.cin.size == 4 * nv.MLP_MAX_LAYERS


def test_parser_reads_the_header_grammar():
    consts, structs, functions = nv.parse_header("""
        #define N_MAX 3  /* bound */
        typedef void* pn_stream_t;
        enum pn_mode { PN_A = 0, PN_B = 1 };
        typedef struct pn_s { int a, b; float c[N_MAX]; const float* p; } pn_s;
        size_t pn_q(void);
        int pn_x(int64_t a, float f, const pn_s* d, const float* const* w, pn_stream_t st);
    """)
    assert consts == {"N_MAX": 3}
    s = structs["pn_s"]
    assert [(f, t) for f, t in s._fields_] == [("a", C.c_int), ("b", C.c_int), ("c", C.c_float * 3), ("p", C.c_void_p)]
    assert functions == {"pn_q": ([], C.c_size_t), "pn_x": ([i64, f32, vp, vp, vp], C.c_int)}


@pytest.mark.parametrize("snippet,names", [
    ("typedef void* pn_stream_t; int pn_x(long double a, pn_stream_t s);", "pn_x"),
    ("double pn_y(int a);", "pn_y"),
    ("int pn_z(int a)", "pn_z"),
    ("int (*pn_cb)(int);", "pn_cb"),
    ("typedef struct pn_t { int a[M]; } pn_t;", "pn_t"),
    ("typedef struct pn_u { int* a, b; } pn_u;", "pn_u"),
])
def test_parser_rejects_what_it_cannot_bind(snippet, names):
    with pytest.raises(ValueError, match=names):
        nv.parse_header(snippet)
