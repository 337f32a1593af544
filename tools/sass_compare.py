"""Check that two builds of libwhvi_b200 compiled the same machine code for every kernel instance of the older one.

    python tools/sass_compare.py OLD_OBJ_DIR NEW_OBJ_DIR [--strip-arg KERNEL ...]

OLD_OBJ_DIR / NEW_OBJ_DIR hold the per-translation-unit objects of ``python -m whvi_b200.build`` (whvi_b200/_obj).  Every
kernel of every object is disassembled with ``cuobjdump -sass`` and keyed by its demangled name (``cu++filt``).  A template
parameter added with a default changes the mangled names of the existing instances, so before the names are matched:
  * ``--strip-dup KERNEL`` drops a trailing type argument of KERNEL when it repeats the one before it (the dx
    type of the backward kernels, which defaults to the activation type: ``<..., float, float>`` and
    ``<..., __nv_bfloat16, __nv_bfloat16>`` are the older ``<..., float>`` and ``<..., __nv_bfloat16>``);
  * ``--strip-arg KERNEL`` then drops a trailing ``, float`` template argument that follows a non-type argument, in both builds
    (default: the four kernels that gained an activation-type parameter for bf16 training, so that builds from before it match);
  * ``--untemplate KERNEL`` keys a kernel that became a template on its element types by its bare name in BOTH builds, where
    every template argument is ``float`` (the plain kernel of the older build); other instances keep their arguments;
  * ``--strip-false KERNEL`` drops a trailing ``, false`` template argument of KERNEL (a ``bool`` flag added last, whose
    ``false`` instances are the older ones) and keys KERNEL's instances without their parameter list, since the flag came
    with extra trailing parameters that the ``false`` instances never read (default: ``categorical_predictive_kernel``, whose
    ``true`` instances add the uncertainty sums, and ``categorical_nll_kernel`` / ``categorical_nll_bwd_kernel``, whose ``true``
    instances take class weights, label smoothing and ignore_index).
Each old instance must have a new instance of the same name whose instructions AND encodings (scheduling control words
included) are identical, line for line; only the instruction addresses are ignored.  New instances without an old counterpart
are listed.  Exit status 1 on any difference.
"""
from __future__ import annotations

import argparse
import re
import subprocess
import sys
from pathlib import Path

CUDA_BIN = Path("/usr/local/cuda/bin")
DEFAULT_STRIP = ("layer_bwd_tma_kernel", "layer_bwd_tm_kernel", "layer_loss_kernel", "layer_loss_tm_kernel")
DEFAULT_STRIP_DUP = ("layer_bwd_tma_kernel", "layer_bwd_tm_kernel")
DEFAULT_UNTEMPLATE = ("stack_split_kernel", "stack_concat_kernel", "stack_sum_kernel", "column_dot_kernel", "column_outer_kernel",
                      "column_dot_dx_kernel", "column_dw_kernel", "column_outer_dx_kernel", "column_dbias_kernel")
DEFAULT_STRIP_FALSE = ("categorical_predictive_kernel", "categorical_nll_kernel", "categorical_nll_bwd_kernel")
_ADDR = re.compile(r"/\*[0-9a-f]{4,}\*/")


def _tool(name: str) -> str:
    p = CUDA_BIN / name
    return str(p) if p.exists() else name


def kernels(obj: Path) -> dict[str, list[str]]:
    """mangled name -> SASS lines (instruction + encoding words, addresses removed)."""
    out = subprocess.run([_tool("cuobjdump"), "-sass", str(obj)], capture_output=True, text=True, check=True).stdout
    funcs: dict[str, list[str]] = {}
    cur = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        if cur is not None and "/*" in line:
            cur.append(" ".join(_ADDR.sub("", line).split()))
    return funcs


def demangle(names: list[str]) -> dict[str, str]:
    if not names:
        return {}
    out = subprocess.run([_tool("cu++filt")], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return dict(zip(names, out.splitlines()))


def normalise(name: str, strip: tuple[str, ...], strip_dup: tuple[str, ...] = (), untemplate: tuple[str, ...] = (),
              strip_false: tuple[str, ...] = ()) -> str:
    for k in strip_false:   # cu++filt prints the flag as ``(bool)0``; the parameter list is dropped too (see --strip-false)
        if re.search(rf"\b{k}<", name):
            name = re.sub(r", (?:false|\(bool\)0)>\(", ">(", name, count=1)
            return name[:name.index(">(") + 1]
    m = re.match(r"(?:void )?whvi::(\w+)(?:<([^()]*)>)?\(", name)
    if m and m.group(1) in untemplate:
        args = m.group(2)
        if args is None or all(a.strip() == "float" for a in args.split(",")):
            return f"whvi::{m.group(1)}"
        return f"whvi::{m.group(1)}<{args}>"
    for k in strip_dup:
        if re.search(rf"\b{k}<", name):
            name = re.sub(r", (float|__nv_bfloat16), \1>\(", r", \1>(", name, count=1)
    for k in strip:   # only a ``float`` that follows a non-type argument: ``<..., __nv_bfloat16, float>`` is a distinct instance
        if re.search(rf"\b{k}<", name):
            return re.sub(r"(\(\w+\)-?\d+), float>\(", r"\1>(", name, count=1)
    return name


def collect(obj_dir: Path, strip: tuple[str, ...], strip_dup: tuple[str, ...] = (), untemplate: tuple[str, ...] = (),
            strip_false: tuple[str, ...] = ()) -> dict[str, tuple[str, list[str]]]:
    res: dict[str, tuple[str, list[str]]] = {}
    for obj in sorted(obj_dir.glob("*.o")):
        funcs = kernels(obj)
        dm = demangle(list(funcs))
        for mangled, sass in funcs.items():
            res[normalise(dm[mangled], strip, strip_dup, untemplate, strip_false)] = (obj.name, sass)
    return res


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("old", type=Path)
    ap.add_argument("new", type=Path)
    ap.add_argument("--strip-arg", nargs="*", default=list(DEFAULT_STRIP))
    ap.add_argument("--strip-dup", nargs="*", default=list(DEFAULT_STRIP_DUP))
    ap.add_argument("--untemplate", nargs="*", default=list(DEFAULT_UNTEMPLATE))
    ap.add_argument("--strip-false", nargs="*", default=list(DEFAULT_STRIP_FALSE))
    a = ap.parse_args()
    untemplate, strip_false = tuple(a.untemplate), tuple(a.strip_false)
    strip, strip_dup = tuple(a.strip_arg), tuple(a.strip_dup)
    old = collect(a.old, strip, strip_dup, untemplate, strip_false)
    new = collect(a.new, strip, strip_dup, untemplate, strip_false)
    same, differ, missing = 0, [], []
    for name, (obj, sass) in sorted(old.items()):
        if name not in new:
            missing.append(f"{obj}: {name}")
        elif new[name][1] != sass:
            differ.append(f"{obj}: {name} ({len(sass)} vs {len(new[name][1])} lines)")
        else:
            same += 1
    added = sorted(f"{obj}: {name}" for name, (obj, _) in new.items() if name not in old)
    print(f"old kernel instances: {len(old)}; identical SASS in the new build: {same}; different: {len(differ)}; "
          f"missing: {len(missing)}; new instances: {len(added)}")
    for title, rows in (("DIFFERENT", differ), ("MISSING", missing), ("new", added)):
        for r in rows:
            print(f"  {title}: {r}")
    return 1 if differ or missing else 0


if __name__ == "__main__":
    sys.exit(main())
