"""CPU: the drop-in boundary without a GPU.  `luaopen_libadcensus` of OUR Lua face (csrc/lua_face.cu built
against oracle/refshim) must register exactly what the reference's own library registers (adcensus.cu:
2061-2105, compiled unmodified; the tables are stored in tests/golden/reference_outputs.json), in the same
order, and argument checking must fail the way luaT does -- all of this happens before any kernel launch, so
no device is needed."""
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FACE = os.path.join(ROOT, "oracle", "_ref", "libadcensus_luaface.so")

pytestmark = pytest.mark.skipif(not os.path.exists(FACE),
                                reason="oracle/_ref not built (python -c 'import __graft_entry__ as g; g.build()')")

HOT = ["StereoJoin", "cross", "cbca", "sgm2", "outlier_detection", "interpolate_occlusion", "interpolate_mismatch",
       "subpixel_enchancement", "median2d", "mean2d", "Normalize_forward", "spatial_argmin", "ad", "census"]


@pytest.fixture(scope="module")
def libs():
    from oracle import reference_outputs, refdriver

    return reference_outputs.load()["functions"], refdriver.ShimLibrary(FACE), refdriver.ShimError


def test_same_tables_as_the_reference(libs):
    ref, face, _ = libs
    assert face.functions("adcensus") == ref["adcensus"]                  # 31 names, registration order included
    assert len(face.functions("adcensus")) == 31
    assert face.functions("nn") == ref["nn"]                              # SpatialLogSoftMax_* (SpatialLogSoftMax.cu:180-189)
    assert set(HOT) <= set(face.functions("adcensus"))


def test_out_of_scope_functions_exist_and_say_so(libs):
    _, face, ShimError = libs
    face.call("version")                                                  # implemented (prints the library version)
    for name in set(face.functions("adcensus")) - set(HOT) - {"version"}:
        with pytest.raises(ShimError, match="not implemented in libadcensus_b200"):
            face.call(name)
    with pytest.raises(ShimError, match="nil value"):                      # what Lua says for a key that was never there
        face.call("no_such_function")


def test_argument_checks_raise_like_luaT(libs):
    _, face, ShimError = libs
    for name in HOT:
        with pytest.raises(ShimError, match="torch.CudaTensor expected"):  # luaT_checkudata on argument 1
            face.call(name, 1.0, 2.0, 3.0, 4.0, 5.0)
