"""development: build a variant of the library whose pxm_fft.cu is compiled with extra -D flags
usage: build_variant.py OUT.so -DFLAG [-DFLAG2 ...] [file.cu]"""
import importlib.util, os, subprocess, sys, tempfile
HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("b", os.path.join(HERE, "pxmcmc_b200", "build.py"))
m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
out = sys.argv[1]
flags = [a for a in sys.argv[2:] if a.startswith("-")]
files = [a for a in sys.argv[2:] if a.endswith(".cu")] or ["pxm_fft.cu"]
bdir = tempfile.mkdtemp()
objs = []
for s in m.SOURCES:
    src = os.path.join(m.CSRC, s)
    if s in files:
        obj = os.path.join(bdir, s.replace(".cu", ".o"))
        r = subprocess.run(["/usr/local/cuda/bin/nvcc", *m.ARCH, *m.COMMON, *m.PER_FILE.get(s, []), *flags, "-c", src, "-o", obj], capture_output=True, text=True)
        if r.returncode:
            sys.exit(r.stderr)
        for line in (r.stdout + r.stderr).splitlines():
            if "fft3_kernel" in line or "fft6_kernel" in line:
                want = True
            elif "Compiling" in line:
                want = False
            if "registers" in line and locals().get("want"):
                print("  ", line.strip())
    else:
        obj = os.path.join(m.HERE, "build", s.replace(".cu", ".o"))
    objs.append(obj)
subprocess.run(["/usr/local/cuda/bin/nvcc", *m.ARCH, "-shared", "-o", out, *objs, "-cudart", "static"], check=True)
print(out)
