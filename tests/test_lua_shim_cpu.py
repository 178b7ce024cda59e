"""CPU suite, part 8: static checks of the LuaJIT shim in lua/ (no Lua interpreter in the image, so the files cannot run
here): every `C.mpn_*` call names a function the header declares and passes as many arguments as its prototype has,
every struct type handed to ffi.new exists in the cdef block, and block keywords balance."""
import glob
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _strip_lua(src):
    src = re.sub(r"--\[\[.*?\]\]", "", src, flags=re.S)
    src = re.sub(r"--[^\n]*", "", src)
    return re.sub(r"'[^'\n]*'", "''", src)


def _split_args(s):
    depth, cur, out = 0, "", []
    for ch in s:
        if ch in "([{":
            depth += 1
        elif ch in ")]}":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur); cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur)
    return out


def _call_args(src, start):
    """text between the parenthesis opening at src[start] and its match"""
    depth = 0
    for i in range(start, len(src)):
        if src[i] == "(":
            depth += 1
        elif src[i] == ")":
            depth -= 1
            if depth == 0:
                return src[start + 1:i]
    raise AssertionError("unbalanced call")


def _prototypes():
    h = open(os.path.join(ROOT, "include", "mpn_abi.h")).read()
    body = re.search(r"MPN_CDEF_BEGIN \*/(.*?)/\* MPN_CDEF_END", h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(mpn_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", body, re.S):
        args = m.group(2).strip()
        protos[m.group(1)] = 0 if args in ("", "void") else len(_split_args(args))
    structs = set(re.findall(r"\}\s*(mpn_[a-z_]+)\s*;", body)) | set(re.findall(r"typedef struct (mpn_[a-z_]+)", body))
    return protos, structs


def test_lua_calls_match_the_header():
    protos, structs = _prototypes()
    assert protos["mpn_nms"] == 6 and protos["mpn_version"] == 0 and "mpn_image_transform" in structs
    files = sorted(glob.glob(os.path.join(ROOT, "lua", "*.lua")))
    assert len(files) >= 5
    seen = set()
    for f in files:
        src = _strip_lua(open(f).read())
        for m in re.finditer(r"\bC\.(mpn_[a-z0-9_]+)\s*\(", src):
            name = m.group(1)
            assert name in protos, f"{os.path.basename(f)} calls {name}, which include/mpn_abi.h does not declare"
            n = len(_split_args(_call_args(src, m.end() - 1)))
            assert n == protos[name], f"{os.path.basename(f)}: {name} called with {n} arguments, prototype has {protos[name]}"
            seen.add(name)
        for m in re.finditer(r"\bC\.(mpn_[a-z0-9_]+)\b(?!\s*\()", src):          # passed as a value (ffi.gc finalizers)
            assert m.group(1) in protos
        for t in re.findall(r"ffi\.new\(''", src):
            pass
    assert {"mpn_nms", "mpn_nms_dense", "mpn_bbox_vote", "mpn_foveal", "mpn_context_region", "mpn_bbox_norm", "mpn_roi_pool",
            "mpn_model_create", "mpn_model_detect", "mpn_model_trunk_image", "mpn_ctx_create"} <= seen
    # struct / pointer types named in ffi.new / ffi.cast strings
    for f in files:
        raw = re.sub(r"--\[\[.*?\]\]", "", open(f).read(), flags=re.S)
        for t in re.findall(r"ffi\.(?:new|cast)\('([^']+)'", raw):
            for ident in re.findall(r"mpn_[a-z_]+", t):
                assert ident in structs or ident in ("mpn_ctx", "mpn_model"), f"{os.path.basename(f)}: unknown C type {ident}"


def test_lua_blocks_balance():
    for f in sorted(glob.glob(os.path.join(ROOT, "lua", "*.lua"))):
        src = _strip_lua(open(f).read())
        depth, pending = 0, 0
        for t in re.findall(r"\b(function|if|for|while|do|end|repeat|until)\b", src):
            if t in ("for", "while"):
                depth += 1; pending += 1
            elif t == "do":
                if pending:
                    pending -= 1
                else:
                    depth += 1
            elif t in ("function", "if", "repeat"):
                depth += 1
            else:
                depth -= 1
            assert depth >= 0, f
        assert depth == 0, f"{os.path.basename(f)}: unbalanced blocks"
        assert src.count("(") == src.count(")") and src.count("{") == src.count("}") and src.count("[") == src.count("]"), f


# ---- the fbcoco.ImageDetect contract (VERDICT r01 item 6): same class, same methods, same argument lists --------------------
IMAGE_DETECT_API = {           # method -> argument names, as ImageDetect.lua:12,91,137,156 declares them
    "__init": ["model", "transformer", "scale", "max_size"],
    "memoryEfficientForward": ["model", "input", "bs", "recompute_features"],
    "computeRawOutputs": ["im", "boxes", "min_images", "recompute_features"],
    "detect": ["im", "boxes", "min_images", "recompute_features"],
}


def _methods(src, cls="ImageDetect"):
    return {m.group(1): [a.strip() for a in m.group(2).split(",") if a.strip()]
            for m in re.finditer(r"function\s+%s:([A-Za-z_]+)\s*\(([^)]*)\)" % cls, src)}


def test_image_detect_keeps_the_reference_contract():
    shim = _strip_lua(open(os.path.join(ROOT, "lua", "ImageDetect_b200.lua")).read())
    assert "torch.class(''" in shim                                      # the class name string was blanked by _strip_lua
    raw = open(os.path.join(ROOT, "lua", "ImageDetect_b200.lua")).read()
    assert "torch.class('fbcoco.ImageDetect')" in raw
    got = _methods(shim)
    assert got == IMAGE_DETECT_API, got
    with open(os.path.join(ROOT, "tests", "golden", "image_detect_api.json")) as f:    # the reference's own table (make_golden.py)
        assert json.load(f) == IMAGE_DETECT_API
    # the constructor keeps the nn module (Tester_FRCNN.lua:37-49 calls module:apply / module:forward / module.output on it)
    assert re.search(r"self\.model\s*=\s*model\b", shim) and "model_desc.create(" in shim
    # no C handle in a serialisable field: the cache is a weak-keyed table, dropped by clearState
    assert re.search(r"handles\s*=\s*setmetatable\(\{\},\s*\{__mode\s*=\s*''\}\)", shim) and "handles[self] = nil" in shim
    assert not re.search(r"self\.[A-Za-z_]*handle\s*=", shim)
    # the CudaTensor path goes through the _dev entry points (no host round trip), the host path through mpn_model_detect
    for fn in ("mpn_model_trunk_dev", "mpn_model_heads_dev", "mpn_model_detect", "mpn_model_trunk_image"):
        assert "C." + fn in shim


def test_tester_fast_path_wraps_without_editing_the_reference_file():
    src = _strip_lua(open(os.path.join(ROOT, "lua", "Tester_b200.lua")).read())
    assert "testOne_reference = Tester.testOne" in src and "function Tester:testOne(i)" in src
    assert "C.mpn_model_detect_nms(" in src and "return testOne_reference(self, i)" in src
    # iterative localisation / rbox scores / voting: one device call as well, with the option struct of the header
    assert "C.mpn_model_test_one(" in src and "ffi.new('mpn_test_opts')" in open(os.path.join(ROOT, "lua", "Tester_b200.lua")).read()
    for field in ("num_iter", "use_rbox_scores", "bbox_voting", "score_thresh", "nms_thr", "vote_thr", "vote_score_pow"):
        assert f"o.{field} =" in src, field
    ffi_src = _strip_lua(open(os.path.join(ROOT, "lua", "mpn_ffi.lua")).read())
    assert "C.mpn_ctx_create_stream(" in ffi_src and "C.mpn_ctx_create(" in ffi_src          # replica streams are opt-in
    mods = _strip_lua(open(os.path.join(ROOT, "lua", "modules_b200.lua")).read())
    assert "C.mpn_roi_pool_dev(" in mods and "C.mpn_roi_pool(" in mods   # CudaTensors stay on the device
