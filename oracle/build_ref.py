#!/usr/bin/env python3
"""Build the UNMODIFIED reference (libjxl 0.13.0) from /root/reference into oracle/_ref/.

TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is on the product path; the
product (libjxl_b200/csrc -> libjxl_b200.so) never links or loads these files.

What this does
--------------
* reads the reference's own source lists (lib/jxl_lists.cmake) at build time,
* compiles every listed .cc **where it lies** under /root/reference with plain
  g++ (no cmake, no ninja, no reference build system), plus the vendored
  Highway / brotli / skcms sources the decoder+encoder need,
* writes the three tiny configuration headers cmake would have produced
  (jxl/version.h, jxl/jxl_export.h, jxl/jxl_cms_export.h, jxl/jxl_threads_export.h)
  into oracle/_ref/include/jxl/,
* archives the objects into oracle/_ref/libjxl_ref.a and links
  oracle/ref_harness.cc (OUR translation unit: a C ABI over the reference's
  internals) into oracle/_ref/libjxl_ref_harness.so.

No reference SOURCE is copied into this repository: outputs are objects, one
archive and one shared library, all under the git-ignored oracle/_ref/.

Flags follow the reference's CMake defaults (lib/CMakeLists.txt:27-137,
CMakeLists.txt:204-238): -O3 -DNDEBUG -fno-rtti -fno-exceptions, Highway
dynamic dispatch with AVX3* / SSSE3 disabled (=> AVX2, SSE4, SSE2 targets, the
"[_AVX2_,SSE4,SSE2]" build SURVEY.md §8c reports), JXL_HIGH_PRECISION default.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import re
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF = Path(os.environ.get("JXL_REFERENCE_ROOT", "/root/reference"))
OUT = HERE / "_ref"
OBJ = OUT / "obj"
INC = OUT / "include"

HWY_DISABLED = "(HWY_AVX3|HWY_AVX3_DL|HWY_AVX3_SPR|HWY_AVX3_ZEN4|HWY_SSSE3)"

COMMON_DEFS = [
    "-DNDEBUG",
    "-DJXL_INTERNAL_LIBRARY_BUILD",
    "-DJXL_STATIC_DEFINE", "-DJXL_CMS_STATIC_DEFINE", "-DJXL_THREADS_STATIC_DEFINE",
    "-DHWY_STATIC_DEFINE",
    "-DJPEGXL_ENABLE_TRANSCODE_JPEG=1", "-DJPEGXL_ENABLE_BOXES=1",
    "-DJPEGXL_ENABLE_SKCMS=1",
    "-DFJXL_ENABLE_AVX512=0",
    f"-DHWY_DISABLED_TARGETS={HWY_DISABLED}",
]
CXXFLAGS = [
    "-std=c++17", "-O3", "-fPIC", "-fno-rtti", "-fno-exceptions",
    "-fmerge-all-constants", "-fno-builtin-fwrite", "-fno-builtin-fread",
    "-fsized-deallocation", "-fmath-errno", "-w", "-pthread",
]
CFLAGS = ["-O2", "-fPIC", "-w"]


def includes() -> list[str]:
    return [
        f"-I{INC}",
        f"-I{REF}",
        f"-I{REF}/lib/include",
        f"-I{REF}/third_party/highway",
        f"-I{REF}/third_party/brotli/c/include",
        f"-I{REF}/third_party/skcms",
    ]


def parse_lists() -> dict[str, list[str]]:
    txt = (REF / "lib" / "jxl_lists.cmake").read_text()
    out: dict[str, list[str]] = {}
    for m in re.finditer(r"set\((\w+)\n(.*?)\n\)", txt, re.S):
        out[m.group(1)] = [l.strip() for l in m.group(2).splitlines() if l.strip()]
    return out


def write_config_headers() -> None:
    (INC / "jxl").mkdir(parents=True, exist_ok=True)
    cm = (REF / "lib" / "CMakeLists.txt").read_text()
    ver = {k: re.search(rf"set\(JPEGXL_{k}_VERSION (\d+)\)", cm).group(1)
           for k in ("MAJOR", "MINOR", "PATCH")}
    tmpl = (REF / "lib" / "jxl" / "version.h.in").read_text()
    for k, v in ver.items():
        tmpl = tmpl.replace(f"@JPEGXL_{k}_VERSION@", v)
    (INC / "jxl" / "version.h").write_text(tmpl)
    for base, fname in (("JXL", "jxl_export.h"), ("JXL_CMS", "jxl_cms_export.h"),
                        ("JXL_THREADS", "jxl_threads_export.h")):
        (INC / "jxl" / fname).write_text(
            f"#ifndef {base}_EXPORT_H\n#define {base}_EXPORT_H\n"
            f"#define {base}_EXPORT __attribute__((visibility(\"default\")))\n"
            f"#define {base}_NO_EXPORT __attribute__((visibility(\"hidden\")))\n"
            f"#define {base}_DEPRECATED __attribute__((__deprecated__))\n"
            f"#endif\n")


def obj_path(src: Path, variant: str) -> Path:
    h = hashlib.sha1(str(src).encode()).hexdigest()[:10]
    return OBJ / variant / f"{src.stem}_{h}.o"


def compile_one(src: Path, extra: list[str], variant: str) -> Path:
    o = obj_path(src, variant)
    if o.exists() and o.stat().st_mtime >= src.stat().st_mtime:
        return o
    if src.suffix == ".c":
        cmd = ["gcc", *CFLAGS, *includes(), *extra, "-c", str(src), "-o", str(o)]
    else:
        cmd = ["g++", *CXXFLAGS, *COMMON_DEFS, *includes(), *extra, "-c", str(src), "-o", str(o)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"compile failed: {' '.join(cmd)}\n{r.stderr[-4000:]}")
    return o


# Two builds of the same sources:
#   default : the reference's own flags (GCC default -ffp-contract=fast lets the
#             compiler fuse Mul+Add pairs of the Highway code into FMAs on its own,
#             so low-order bits are compiler dependent) -> CPU baseline timing and
#             image-level oracle.
#   strict  : adds -ffp-contract=off, i.e. FMAs exactly where the source says
#             MulAdd/NegMulAdd -> bit-exact pin for oracle/jxl_oracle.c.
VARIANTS = {"default": ("libjxl_ref_harness.so", []),
            "strict": ("libjxl_ref_harness_strict.so", ["-ffp-contract=off"])}

# A third library, "gpu": the reference with the jxl_b200 backend compiled in (INTEGRATION.md §2) -- the
# same objects as "default" except lib/jxl/dec_frame.cc and lib/jxl/dec_group.cc, which are built from the
# patched copies integration/patch_libjxl.py writes to oracle/_ref/patched/ (hooks into OUR
# integration/libjxl_gpu_backend.h), linked against libjxl_b200/libjxl_b200.so.  It is what measures
# T_e2e (.jxl bytes -> pixels through the public JxlDecoder API with the GPU doing the transform path).
GPU_SO = "libjxl_ref_harness_gpu.so"
PATCHED = ("lib/jxl/dec_frame.cc", "lib/jxl/dec_group.cc")


def reference_present() -> bool:
    """The reference source tree is there and readable (a tree under a directory this user may not enter
    counts as absent)."""
    return os.access(REF / "lib" / "jxl_lists.cmake", os.R_OK)


def main() -> int:
    if not reference_present():
        print(f"[build_ref] {REF} not present: keeping prebuilt oracle/_ref as is")
        return 0 if (OUT / "libjxl_ref_harness.so").exists() else 1
    write_config_headers()
    for variant in VARIANTS:
        rc = build_variant(variant)
        if rc:
            return rc
    return build_gpu_variant()


def build_gpu_variant() -> int:
    product = HERE.parent / "libjxl_b200" / "libjxl_b200.so"
    if not product.exists():
        print("[build_ref] [gpu] libjxl_b200.so not built yet: skipping the integrated variant")
        return 0
    repo = HERE.parent
    patched_dir = OUT / "patched"
    subprocess.check_call([sys.executable, str(repo / "integration" / "patch_libjxl.py"), str(REF), str(patched_dir)])
    (OBJ / "gpu").mkdir(parents=True, exist_ok=True)
    extra = [f"-I{repo / 'integration'}", f"-I{repo / 'include'}"]
    hdrs = [repo / "integration" / n for n in ("libjxl_gpu_backend.h", "gpu_frame_binding.h", "pinned_ac_image.h")]
    hdrs.append(repo / "include" / "jxl_b200.h")
    new_objs = {}
    for rel in PATCHED:
        src = patched_dir / rel
        o = OBJ / "gpu" / (Path(rel).stem + ".o")
        if not (o.exists() and o.stat().st_mtime >= max([src.stat().st_mtime] + [h.stat().st_mtime for h in hdrs])):
            # the patched tree first: dec_group.cc re-includes itself per Highway target (see patch_libjxl.py)
            cmd = ["g++", *CXXFLAGS, *COMMON_DEFS, f"-I{patched_dir}", *includes(), *extra, "-c", str(src), "-o", str(o)]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"compile failed: {' '.join(cmd)}\n{r.stderr[-6000:]}")
        new_objs[str(REF / rel)] = o
    # every other object is the default variant's
    objs = []
    for s_, _ in source_list([]):
        objs.append(new_objs.get(str(s_), obj_path(s_, "default")))
    lib = OUT / "libjxl_ref_gpu.a"
    if lib.exists():
        lib.unlink()
    subprocess.check_call(["ar", "rcs", str(lib), *map(str, objs)])
    so = OUT / GPU_SO
    cmd = ["g++", *CXXFLAGS, *COMMON_DEFS, "-DJXLB_REF_HARNESS_GPU=1", *includes(), f"-I{repo / 'include'}", *extra,
           "-shared", str(HERE / "ref_harness.cc"),
           "-Wl,--whole-archive", str(lib), "-Wl,--no-whole-archive", "-Wl,--exclude-libs,ALL",
           f"-L{product.parent}", "-l:libjxl_b200.so", "-Wl,-rpath,$ORIGIN/../../libjxl_b200",
           "-lpthread", "-lm", "-o", str(so)]
    cmd.remove("-w")
    cmd.append("-Wno-attributes")
    subprocess.check_call(cmd)
    print(f"[build_ref] built {so}")
    return 0


def source_list(vflags: list[str]) -> list[tuple[Path, list[str]]]:
    """Every reference / vendored source of the library with its extra flags, de-duplicated."""
    lists = parse_lists()
    srcs: list[tuple[Path, list[str]]] = []
    for key in ("JPEGXL_INTERNAL_BASE_SOURCES", "JPEGXL_INTERNAL_DEC_SOURCES",
                "JPEGXL_INTERNAL_DEC_BOX_SOURCES", "JPEGXL_INTERNAL_DEC_JPEG_SOURCES",
                "JPEGXL_INTERNAL_ENC_SOURCES", "JPEGXL_INTERNAL_CMS_SOURCES",
                "JPEGXL_INTERNAL_THREADS_SOURCES"):
        for f in lists[key]:
            if f.endswith(".cc"):
                srcs.append((REF / "lib" / f, []))
    # function-level facade the reference's own ac_strategy_test uses
    # (lib/jxl/dec_transforms_testonly.h:20-30)
    srcs.append((REF / "lib/jxl/dec_transforms_testonly.cc", []))
    srcs.append((REF / "lib/jxl/enc_transforms.cc", []))
    for f in ("abort.cc", "aligned_allocator.cc", "per_target.cc", "print.cc",
              "targets.cc", "timer.cc"):
        srcs.append((REF / "third_party/highway/hwy" / f, []))
    for sub in ("common", "dec", "enc"):
        for f in sorted((REF / "third_party/brotli/c" / sub).glob("*.c")):
            srcs.append((f, []))
    skdefs = ["-DSKCMS_DISABLE_HSW", "-DSKCMS_DISABLE_SKX", "-Wno-psabi"]
    srcs = [(s_, e_ + vflags) for s_, e_ in srcs]
    skdefs = skdefs + vflags
    srcs.append((REF / "third_party/skcms/skcms.cc", skdefs))
    srcs.append((REF / "third_party/skcms/src/skcms_TransformBaseline.cc", skdefs))
    # de-duplicate (enc_transforms.cc is already in the ENC list)
    seen, uniq = set(), []
    for s, e in srcs:
        if s not in seen:
            seen.add(s)
            uniq.append((s, e))
    return uniq


def build_variant(variant: str) -> int:
    so_name, vflags = VARIANTS[variant]
    (OBJ / variant).mkdir(parents=True, exist_ok=True)
    uniq = source_list(vflags)
    jobs = int(os.environ.get("JOBS", os.cpu_count() or 4))
    print(f"[build_ref] [{variant}] compiling {len(uniq)} reference sources with {jobs} jobs")
    objs = []
    with cf.ThreadPoolExecutor(jobs) as ex:
        futs = [ex.submit(compile_one, s, e, variant) for s, e in uniq]
        for i, f in enumerate(futs):
            objs.append(f.result())
            if (i + 1) % 40 == 0:
                print(f"[build_ref]   {i + 1}/{len(uniq)}")
    lib = OUT / f"libjxl_ref_{variant}.a"
    if lib.exists():
        lib.unlink()
    subprocess.check_call(["ar", "rcs", str(lib), *map(str, objs)])
    harness = HERE / "ref_harness.cc"
    so = OUT / so_name
    cmd = ["g++", *CXXFLAGS, *vflags, *COMMON_DEFS, *includes(), f"-I{HERE.parent / 'include'}", "-shared", str(harness),
           "-Wl,--whole-archive", str(lib), "-Wl,--no-whole-archive",
           "-Wl,--exclude-libs,ALL", "-lpthread", "-lm", "-o", str(so)]
    cmd.remove("-w")
    cmd.append("-Wno-attributes")
    subprocess.check_call(cmd)
    print(f"[build_ref] built {so}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
