"""Compare the machine code of two versions of one CUDA source of the library (no GPU needed).

    python bench_micro/sass_diff.py OLD.cu NEW.cu

Both files are compiled with the library's flags (``__graft_entry__.NVCC_FLAGS``, the library's include
directories, ``-Xptxas -v``), dumped with ``cuobjdump -sass`` and split per function, with the ``/*0x....*/``
address comments stripped.  Prints every function whose instructions or ptxas resource line (registers, shared
memory, spills) differ, and functions present on one side only; exits 1 if there is any difference.
To compare against a commit: ``git show REV:climate_toolbox_b200/csrc/ctb_plan.cu > /tmp/old.cu``."""
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import NVCC_FLAGS  # noqa: E402

NVCC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
CUOBJDUMP = os.path.join(os.path.dirname(NVCC), "cuobjdump")


def _name(mangled):
    """The anonymous namespace's tag depends on the source file, not on the kernel: drop it."""
    return re.sub(r"\d+_GLOBAL__N__\w+?_[0-9a-f]{8}", "(anon)", mangled)


def compile_one(src, tmp, tag):
    obj = os.path.join(tmp, tag + ".o")
    cmd = [NVCC] + NVCC_FLAGS + ["-Xptxas", "-v", "-I", os.path.join(ROOT, "include"),
                                 "-I", os.path.join(ROOT, "climate_toolbox_b200", "csrc"), "-c", src, "-o", obj]
    log = subprocess.run(cmd, check=True, capture_output=True, text=True).stderr
    # ptxas -v: "Compiling entry function '<name>'" ... "Used N registers, ..." per kernel
    res, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = _name(m.group(1))
        elif cur and ("spill" in line or "Used" in line):
            res[cur] = res.get(cur, "") + re.sub(r"^.*?: ", "", line.strip()) + " | "
    sass = subprocess.run([CUOBJDUMP, "-sass", obj], check=True, capture_output=True, text=True).stdout
    funcs, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = _name(m.group(1))
            funcs[cur] = []
        elif cur and "/*" in line:
            ins = re.sub(r"/\*[0-9a-fx]+\*/", "", line).strip()
            if ins:
                funcs[cur].append(ins)
    return funcs, res


def main(old, new):
    with tempfile.TemporaryDirectory() as tmp:
        (fa, ra), (fb, rb) = compile_one(old, tmp, "old"), compile_one(new, tmp, "new")
    diff = 0
    for name in sorted(set(fa) | set(fb)):
        if name not in fa or name not in fb:
            print("only in {}: {}".format("old" if name in fa else "new", name))
            diff += 1
        elif fa[name] != fb[name] or ra.get(name) != rb.get(name):
            print("differs: {}\n  old: {}\n  new: {}".format(name, ra.get(name), rb.get(name)))
            diff += 1
    print("{} functions, {} differ".format(len(set(fa) | set(fb)), diff))
    for name in sorted(fb):
        print("  {}  {}".format(rb.get(name, "-"), name))
    return 1 if diff else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
