"""Per-kernel SASS fingerprint of a shared library, for checking that a host-side change left the device code as it
was: python tools/sass_fp.py lib.so > fp.txt, once per build, then diff the two files.

Each line is the hash of one kernel body and the kernel's name.  The body is normalised so that only the
instructions count: address columns, column padding, blank lines and the fatbin / ELF section lines are dropped,
and the per-translation-unit hash in anonymous-namespace names is replaced by a fixed string.  A kernel that moves to
another translation unit therefore keeps its fingerprint."""
import hashlib, re, subprocess, sys
out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", sys.argv[1]], capture_output=True, text=True, check=True).stdout
funcs, name, body = {}, None, []
skip = re.compile(r"\s*($|(identifier|code for|code version|compressed|Fatbin|arch|host|compile_size|producer)\b|\.(target|headerflags)\b|=+\s*$)")
for line in out.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        if name: funcs.setdefault(name, []).append("\n".join(body))
        name, body = m.group(1), []
    elif name and not skip.match(line):
        body.append(" ".join(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).split()))
if name: funcs.setdefault(name, []).append("\n".join(body))
for n in sorted(funcs):
    for b in funcs[n]:
        print(hashlib.sha256(b.encode()).hexdigest()[:16], re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", n))
