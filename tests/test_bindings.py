"""The reference-side binding (INTEGRATION.md): the N-API shim must compile against the C ABI header (syntax check
with the minimal N-API declarations — there is no Node in the image), call only functions include/bbq_b200.h declares,
and the TypeScript class must call only functions the shim registers."""
import os
import re
import subprocess

from tests.golden_util import REFERENCE_DIR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAPI = os.path.join(ROOT, "better-binary-quantization_b200", "bindings", "napi")
TS = os.path.join(ROOT, "better-binary-quantization_b200", "bindings", "ts")


def test_napi_shim_compiles_against_the_header():
    out = subprocess.run(["gcc", "-fsyntax-only", "-Wall", "-Werror", "-I", NAPI, "-I", os.path.join(ROOT, "include"),
                          os.path.join(NAPI, "bbq_napi.c")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr


def test_shim_calls_only_declared_entry_points():
    header = open(os.path.join(ROOT, "include", "bbq_b200.h")).read()
    declared = set(re.findall(r"\b(bbq_[a-z_0-9]+)\s*\(", header))
    shim = open(os.path.join(NAPI, "bbq_napi.c")).read()
    called = set(re.findall(r"\b(bbq_[a-z_0-9]+)\s*\(", shim))
    assert called and called <= declared, called - declared
    # the path's entry points are all reachable from JavaScript
    for fn in ("bbq_create", "bbq_index_build", "bbq_search", "bbq_index_export", "bbq_index_attach_rows",
               "bbq_search_rerank", "bbq_index_save", "bbq_index_load", "bbq_destroy", "bbq_index_destroy",
               "bbq_quantize_query", "bbq_quantization_accuracy", "bbq_index_from_quantized", "bbq_search_sharded",
               "bbq_comm_unique_id", "bbq_comm_init", "bbq_index_set_base"):
        assert fn in called, fn


def test_typescript_class_uses_registered_addon_functions():
    shim = open(os.path.join(NAPI, "bbq_napi.c")).read()
    registered = set(re.findall(r'\{"([A-Za-z]+)", NULL, n_', shim))
    ts = open(os.path.join(TS, "binaryQuantizationFormat.gpu.ts")).read()
    used = set(re.findall(r"\baddon\.([A-Za-z]+)\(", ts))
    assert used and used <= registered, used - registered
    for name in ("dimension()", "size()", "getCentroid", "vectorValue", "getUnpackedVector", "getCorrectiveTerms"):
        assert name in ts, name      # src/types.ts:32-49


REFERENCE_CLASS = os.path.join(REFERENCE_DIR, "src", "binaryQuantizationFormat.ts") if REFERENCE_DIR else ""
# the ten public members of the reference class, src/binaryQuantizationFormat.ts:141-601
PUBLIC_MEMBERS = ["constructor", "quantizeVectors", "quantizeQueryVector", "searchNearestNeighbors",
                  "computeQuantizationAccuracy", "serializeVectorData", "deserializeVectorData", "getConfig",
                  "getQuantizer", "getScorer"]


def test_typescript_class_keeps_every_public_member_of_the_reference():
    """The replacement class must type-check wherever the reference class did (src/index.ts:133 calls
    computeQuantizationAccuracy): it EXTENDS the reference class, overrides the members on the path with the
    reference's exact signatures, and inherits the three accessors."""
    ts = open(os.path.join(TS, "binaryQuantizationFormat.gpu.ts")).read()
    assert re.search(r"export class BinaryQuantizationFormat extends ReferenceBinaryQuantizationFormat", ts)
    assert "from './binaryQuantizationFormat.cpu'" in ts
    overridden = set(re.findall(r"public override (\w+)\(", ts))
    assert overridden == {"quantizeVectors", "quantizeQueryVector", "searchNearestNeighbors",
                          "computeQuantizationAccuracy", "serializeVectorData", "deserializeVectorData"}
    assert "constructor(config: BinaryQuantizationConfig)" in ts and "super(config)" in ts
    inherited = set(PUBLIC_MEMBERS) - overridden - {"constructor"}
    assert inherited == {"getConfig", "getQuantizer", "getScorer"}
    if REFERENCE_CLASS and os.path.exists(REFERENCE_CLASS):   # with a reference checkout (BBQ_REFERENCE_DIR)
        ref = open(REFERENCE_CLASS, encoding="utf-8").read()
        body = ref[ref.index("export class BinaryQuantizationFormat"):]
        ref_public = set(re.findall(r"^  public (\w+)\(", body, flags=re.M)) | {"constructor"}
        assert ref_public == set(PUBLIC_MEMBERS), ref_public ^ set(PUBLIC_MEMBERS)
        # same parameter lists as the reference for every overridden member
        for name in overridden:
            want = re.search(rf"public {name}\(([^)]*)\)", body, flags=re.S).group(1)
            got = re.search(rf"public override {name}\(([^)]*)\)", ts, flags=re.S).group(1)
            norm = lambda t: re.sub(r"\s+", "", t)
            assert norm(got) == norm(want), (name, got, want)


def test_error_table_covers_every_reference_status():
    errors = open(os.path.join(TS, "errors.ts")).read()
    header = open(os.path.join(ROOT, "include", "bbq_b200.h")).read()
    for status in range(1, 9):   # the statuses that stand for a `throw new Error(...)` of the reference
        assert re.search(rf"BBQ_ERR_[A-Z_]+ = {status},", header), status
        assert f"case {status}:" in errors, status
