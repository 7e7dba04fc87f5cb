"""Drop-in boundary checks that need no GPU: the product library loads, exports every symbol that
include/embree4_b200.h declares, the POD layouts equal the reference's (measured values from SURVEY 8b and the
same probe compiled against the reference headers, tests/golden/reference_abi.json), and the library fails loudly --
it has no CPU fallback -- when no CUDA device exists."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "embree4_b200.h")
LIB = os.path.join(ROOT, "embree_b200", "csrc", "libembree4_b200.so")

PROBE = r"""
#include <stdio.h>
#include <stddef.h>
#include HEADER
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n",
    sizeof(struct RTCRay), sizeof(struct RTCHit), sizeof(struct RTCRayHit), offsetof(struct RTCRayHit, hit),
    sizeof(struct RTCRayHit4), sizeof(struct RTCRayHit8), sizeof(struct RTCRayHit16), sizeof(struct RTCRay16),
    offsetof(struct RTCRayHit16, hit), offsetof(struct RTCHit, primID), offsetof(struct RTCRay, tfar),
    sizeof(struct RTCBounds), sizeof(struct RTCIntersectArguments), sizeof(struct RTCRayQueryContext));
  printf("%d %d %d %d %d %d\n", (int)RTC_FORMAT_FLOAT3, (int)RTC_FORMAT_UINT3, (int)RTC_BUFFER_TYPE_VERTEX,
    (int)RTC_ERROR_INVALID_OPERATION, (int)RTC_RAY_QUERY_FLAG_COHERENT, (int)RTC_DEVICE_PROPERTY_RAY_MASK_SUPPORTED);
  /* callback / interpolation argument blocks and the curve, filter and tangent enumerators added in round 2 */
  printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(struct RTCFilterFunctionNArguments), offsetof(struct RTCFilterFunctionNArguments, hit),
    offsetof(struct RTCFilterFunctionNArguments, N), sizeof(struct RTCInterpolateArguments), offsetof(struct RTCInterpolateArguments, P),
    sizeof(struct RTCInterpolateNArguments), offsetof(struct RTCInterpolateNArguments, valueCount));
  printf("%d %d %d %d %d %d %d %d %d %d %d %d\n", (int)RTC_GEOMETRY_TYPE_FLAT_BEZIER_CURVE, (int)RTC_GEOMETRY_TYPE_ROUND_BEZIER_CURVE,
    (int)RTC_GEOMETRY_TYPE_FLAT_BSPLINE_CURVE, (int)RTC_GEOMETRY_TYPE_ROUND_BSPLINE_CURVE, (int)RTC_GEOMETRY_TYPE_FLAT_HERMITE_CURVE,
    (int)RTC_GEOMETRY_TYPE_ROUND_HERMITE_CURVE, (int)RTC_GEOMETRY_TYPE_FLAT_CATMULL_ROM_CURVE, (int)RTC_GEOMETRY_TYPE_ROUND_CATMULL_ROM_CURVE,
    (int)RTC_BUFFER_TYPE_TANGENT, (int)RTC_RAY_QUERY_FLAG_INVOKE_ARGUMENT_FILTER, (int)RTC_FEATURE_FLAG_FLAT_BEZIER_CURVE,
    (int)RTC_FEATURE_FLAG_ROUND_CATMULL_ROM_CURVE);
  printf("%d %d %d %d %d %d %d %d\n", (int)RTC_GEOMETRY_TYPE_SPHERE_POINT, (int)RTC_GEOMETRY_TYPE_DISC_POINT, (int)RTC_GEOMETRY_TYPE_ORIENTED_DISC_POINT,
    (int)RTC_BUFFER_TYPE_NORMAL, (int)RTC_FEATURE_FLAG_SPHERE_POINT, (int)RTC_FEATURE_FLAG_DISC_POINT, (int)RTC_FEATURE_FLAG_ORIENTED_DISC_POINT,
    (int)RTC_DEVICE_PROPERTY_POINT_GEOMETRY_SUPPORTED);
  return 0;
}
"""


def _probe(header_path, extra_inc=()):
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "p.c")
        open(src, "w").write(PROBE.replace("HEADER", f'"{header_path}"'))
        exe = os.path.join(d, "p")
        subprocess.check_call(["gcc", "-std=gnu11", "-o", exe, src] + [f"-I{i}" for i in extra_inc])
        return subprocess.check_output([exe]).decode().split()


def test_layout_matches_reference_values():
    got = _probe(HEADER)
    # sizeof(RTCRay)=48, RTCHit=48, RTCRayHit=96, offsetof(hit)=48, RTCRayHit4/8/16 = 336/672/1344 (SURVEY 8b, measured)
    assert got[:7] == ["48", "48", "96", "48", "336", "672", "1344"]
    assert got[7] == "768" and got[8] == "768"
    assert got == _reference_abi()["layout_probe"]   # the same probe compiled against the reference's headers


def _reference_abi():
    """tests/golden/reference_abi.json (make_golden.py abi): the probe's output and every rtc* prototype of the reference headers."""
    import json
    return json.load(open(os.path.join(ROOT, "tests", "golden", "reference_abi.json")))


def _declared_symbols():
    txt = open(HEADER).read()
    names = set(re.findall(r"RTCB200_API[^;(]*?\b(rtc\w+)\s*\(", txt))
    names |= set(re.findall(r"RTCB200_DECLARE_UNSUPPORTED\((rtc\w+)\)", txt))
    return sorted(names)


def test_library_exports_every_declared_symbol():
    assert os.path.exists(LIB), "build the library first: python -c 'import __graft_entry__ as g; g.build()'"
    names = _declared_symbols()
    assert len(names) > 80
    out = subprocess.check_output(["nm", "-D", "--defined-only", LIB]).decode()
    exported = set(l.split()[-1] for l in out.splitlines() if " T " in l)
    missing = [n for n in names if n not in exported]
    assert not missing, missing
    dll = C.CDLL(LIB)
    for n in names:
        getattr(dll, n)


def test_every_reference_export_is_present():
    """Any Embree 4 caller links: every rtc* symbol the unmodified reference library exports (list in
    tests/reference_exports.txt, taken with nm -D from oracle/_ref) is exported here too; unsupported ones report
    RTC_ERROR_INVALID_OPERATION when called."""
    want = [l.strip() for l in open(os.path.join(ROOT, "tests", "reference_exports.txt")) if l.strip() and not l.startswith("#")]
    assert len(want) >= 150
    ref_so = os.path.join(ROOT, "oracle", "_ref", "libembree4.so.4")
    if os.path.exists(ref_so):   # the committed list is what the reference build really exports
        out = subprocess.check_output(["nm", "-D", "--defined-only", ref_so]).decode()
        live = sorted(set(l.split()[-1] for l in out.splitlines() if l.split()[-1].startswith("rtc")))
        assert live == sorted(want)
    out = subprocess.check_output(["nm", "-D", "--defined-only", LIB]).decode()
    have = set(l.split()[-1] for l in out.splitlines())
    assert not [w for w in want if w not in have]
    dll = C.CDLL(LIB)
    dll.rtcGetDeviceError.argtypes = [C.c_void_p]
    dll.rtcGetDeviceError(None)
    dll.rtcNewBVH.restype = C.c_void_p
    assert dll.rtcNewBVH(None) is None
    assert dll.rtcGetDeviceError(None) == 3     # RTC_ERROR_INVALID_OPERATION
    assert dll.rtcGetDeviceError(None) == 0


def test_only_rtc_symbols_and_sm100a_code():
    """Nothing but the C-ABI is exported, and the embedded device code is sm_100a only."""
    out = subprocess.check_output(["nm", "-D", "--defined-only", LIB]).decode()
    funcs = [l.split()[-1] for l in out.splitlines() if " T " in l]
    stray = [f for f in funcs if not f.startswith("rtc") and not f.startswith("_")]
    assert not stray, stray
    cu = subprocess.run(["cuobjdump", "-lelf", LIB], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", cu))
    assert archs == {"sm_100a"}, archs


def test_fails_loudly_without_a_gpu():
    """No CPU fallback: on a machine without CUDA, rtcNewDevice returns NULL and reports why."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import embree_b200
    lib = embree_b200.load()
    d = lib.rtcNewDevice(None)
    assert not d
    assert lib.rtcGetDeviceError(None) == 1  # RTC_ERROR_UNKNOWN
    assert b"CUDA" in lib.rtcGetDeviceLastErrorMessage(None)


def test_error_strings():
    import embree_b200
    lib = embree_b200.load()
    assert lib.rtcGetErrorString(0) == b"No error"
    assert lib.rtcGetErrorString(3) == b"Invalid operation"


def _prototypes(text):
    """{function name: (return type, [parameter types])} of every rtc* declaration in a header; types are compared modulo
    struct / enum / const keywords, parameter names and export macros."""
    import re
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"//[^\n]*", "", text)
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)
    text = re.sub(r"\s+", " ", text)
    macros = r"\b(RTC_API|RTC_API_EXTERN_C|RTC_SYCL_API|RTCB200_API|RTC_SYCL_INDIRECTLY_CALLABLE|RTC_FORCEINLINE|RTC_OPTIONAL_ARGUMENT|extern|struct|enum|const)\b"
    out = {}
    for m in re.finditer(r"([A-Za-z_][A-Za-z0-9_ \*]*?)\b(rtc[A-Z][A-Za-z0-9]*)\s*\(([^;{]*?)\)\s*;", text):
        ret = re.sub(macros, "", m.group(1)).replace(" ", "")
        params = []
        for a in (m.group(3).split(",") if m.group(3).strip() else []):
            a = re.sub(r"\s+", " ", re.sub(macros, "", a)).strip()
            named = re.match(r"^(.*?)([A-Za-z_][A-Za-z0-9_]*)$", a)
            if named and named.group(1).strip():
                a = named.group(1)
            params.append(a.replace(" ", ""))
        out[m.group(2)] = (ret, params)
    return out


def test_prototypes_match_the_reference_headers():
    """Every rtc* function include/embree4_b200.h declares has the reference's signature (return type, parameter types and order,
    include/embree4/rtcore_*.h); the reference functions the header does not declare are exactly the stubs outside the path."""
    ref = {n: (r, p) for n, (r, p) in _reference_abi()["prototypes"].items()}
    mine = _prototypes(open(HEADER).read())
    shared = [n for n in mine if n in ref]
    assert len(shared) >= 85
    wrong = {n: (ref[n], mine[n]) for n in shared if ref[n] != mine[n]}
    assert not wrong, wrong
    undeclared = set(ref) - set(mine)
    unsupported = ("Forward", "PointQuery", "BVH", "Collide", "HalfEdge", "GeometryFace", "SYCL", "WithQueue", "InvokeIntersectFilter",
                   "InvokeOccludedFilter", "BoundsFunction", "DisplacementFunction", "InstancedScenes", "IntersectFunction", "OccludedFunction",
                   "PointQueryFunction", "Subdivision", "Topology", "TransformQuaternion", "UserPrimitiveCount", "ThreadLocalAlloc")
    assert all(any(u in n for u in unsupported) for n in undeclared), sorted(n for n in undeclared if not any(u in n for u in unsupported))
