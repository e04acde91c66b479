"""CPU tests: the C-ABI library loads and exports every symbol include/geopolars_b200.h declares
(no compute without a GPU), the product fails loudly without a device, and the host-side logic."""
import os
import re

import numpy as np
import pytest

from geopolars_b200 import GeoArrowArray, GeometryType, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "geopolars_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gpl_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 45
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported by libgeopolars_b200.so"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature in geopolars_b200/_lib.py"
    assert set(_lib.SIGNATURES) <= set(names)
    assert lib.gpl_abi_version() == 1


def test_no_cpu_fallback_without_a_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from geopolars_b200.engine import Context

    with pytest.raises(_lib.GeopolarsError) as e:
        Context(0)
    assert "no CPU fallback" in str(e.value)


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "geopolars_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                for line in open(os.path.join(dirpath, f), errors="replace"):
                    code = line.split("//")[0].split("#", 1)[0] if f.endswith(".py") else line.split("//")[0]
                    if f.endswith(".py"):
                        assert not re.search(r"\b(import|from)\s+oracle\b", code), (f, line)
                    else:
                        assert not (code.lstrip().startswith("#include") and "oracle" in code), (f, line)
                    assert "libgeo_oracle" not in code, (f, line)


def test_library_reads_no_environment():
    """the library's behaviour is a function of its inputs: no kernel variant or tuning value is chosen by an environment
    variable (another build is compared by loading it through GEOPOLARS_B200_LIB instead)"""
    csrc = os.path.join(ROOT, "geopolars_b200", "csrc")
    sources = [f for f in os.listdir(csrc) if f.endswith((".cu", ".cuh", ".cpp", ".h")) or f == "Makefile"]
    assert "k_pip.cu" in sources
    for f in sources:
        assert "getenv" not in open(os.path.join(csrc, f), errors="replace").read(), f


def test_geoarrow_container_and_row_sharding():
    sq = [(0, 0), (1, 0), (1, 1), (0, 1), (0, 0)]
    mp = GeoArrowArray.from_shapes(GeometryType.MULTIPOLYGON, [[[sq], [sq, sq]], [], [[sq]], None])
    assert len(mp) == 4 and mp.n_parts == 3 and mp.n_rings == 4 and mp.n_coords == 20
    assert mp.valid.tolist() == [True, True, True, False]
    part = mp.take_rows(2, 4)
    assert len(part) == 2 and part.geom_off.tolist() == [0, 1, 1] and part.ring_off.tolist() == [0, 5]
    assert np.array_equal(part.xy, np.array(sq, float))
    with pytest.raises(ValueError):
        GeoArrowArray(GeometryType.POLYGON, np.zeros((0, 2)))
    from geopolars_b200 import engine

    assert engine._origin("Centroid")[0] == 0 and engine._origin((1, 2)) == (2, 1.0, 2.0) and engine._origin({"x": 3, "y": 4})[1:] == (3.0, 4.0)
    with pytest.raises(ValueError):
        engine._origin("middle")


def test_rust_shim_is_complete_and_binds_declared_symbols():
    """bindings/geoseries_b200.rs (the source a maintainer drops next to geoseries.rs): every method of the reference trait
    (geopolars/geopolars-geo/src/geoseries.rs:10-181) is implemented, and every extern "C" fn it declares is declared by
    include/geopolars_b200.h with the same number of parameters."""
    rs = open(os.path.join(ROOT, "bindings", "geoseries_b200.rs")).read()
    trait_methods = ["affine_transform", "area", "centroid", "convex_hull", "envelope", "euclidean_length", "exterior", "explode",
                     "geodesic_length", "geom_type", "is_empty", "is_ring", "rotate", "scale", "simplify", "skew", "distance",
                     "to_crs", "to_crs_with_options", "translate", "x", "y"]
    impl = rs[rs.index("impl GeoSeries for Series"):rs.index("pub trait GeoSeriesB200Ext")]
    for m in trait_methods:
        assert re.search(r"\bfn %s\(" % m, impl), f"trait method {m} missing from the Rust shim"
    assert "todo!" not in rs and "unimplemented!" not in rs
    hdr = open(os.path.join(ROOT, "include", "geopolars_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    block = rs[rs.index('extern "C" {'):]
    block = block[:block.index("\n}")]
    for name, params in re.findall(r"fn (gpl_[a-z0-9_]+)\((.*?)\)", block, flags=re.S):
        m = re.search(r"\b%s\s*\((.*?)\)" % name, hdr, flags=re.S)
        assert m, f"{name} is bound by the Rust shim but not declared in the header"
        n_rs = 0 if not params.strip() else params.count(",") + 1
        c_params = m.group(1).strip()
        n_c = 0 if c_params in ("", "void") else c_params.count(",") + 1
        assert n_rs == n_c, f"{name}: {n_rs} parameters in the Rust shim, {n_c} in the header"


def test_bundled_datasets_are_arrow_ipc_files():
    import pyarrow.ipc as ipc

    from geopolars_b200 import datasets

    rows = {"naturalearth_cities": 243, "nybb": 5, "naturalearth_lowres": 177, "cities": 202}
    for name in datasets.available:
        with open(datasets.get_path(name), "rb") as f:
            t = ipc.open_file(f).read_all()
        assert t.num_rows == rows[name] and t.schema.field("geometry").type == "binary"
    with pytest.raises(ValueError):
        datasets.get_path("nope")


def test_accessor_mirrors_the_reference_surface():
    """every entry point of the reference's `.geo` accessor (py-geopolars/python/geopolars/internals/georust/geoseries.py:22-309)
    and every method of its Rust trait (geopolars/geopolars-geo/src/geoseries.rs:10-181) exists under the same name, as a
    property where the reference has a property, with the reference's parameter names and defaults"""
    import inspect

    from geopolars_b200.geoseries import GeoRustSeries

    properties = ["area", "centroid", "geom_type", "x", "y"]
    methods = {
        "affine_transform": ["matrix"], "convex_hull": [], "envelope": [], "euclidean_length": [], "exterior": [],
        "geodesic_length": ["method"], "is_empty": [], "is_ring": [], "rotate": ["angle", "origin"], "scale": ["xfact", "yfact", "origin"],
        "skew": ["xs", "ys", "origin"], "distance": ["other"], "translate": ["xoff", "yoff"],
        # trait methods the Python accessor of the reference does not expose yet (geoseries.rs:47-53, 126-139)
        "explode": [], "simplify": ["tolerance"],
    }
    for p in properties:
        assert isinstance(inspect.getattr_static(GeoRustSeries, p), property), p
    for name, params in methods.items():
        fn = inspect.getattr_static(GeoRustSeries, name)
        assert callable(fn) and not isinstance(fn, property), name
        assert list(inspect.signature(fn).parameters)[1:] == params, (name, list(inspect.signature(fn).parameters))
    sig = inspect.signature(GeoRustSeries.rotate)
    assert sig.parameters["origin"].default == "center"  # georust/geoseries.py:187
    assert inspect.signature(GeoRustSeries.geodesic_length).parameters["method"].default == "geodesic"  # :128
    assert inspect.signature(GeoRustSeries.translate).parameters["xoff"].default == 0.0  # :278
