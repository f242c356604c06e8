"""Build libsnb200.so (sm_100a only) in-tree with nvcc.  Usage: python build.py [--force] [--example [OUT]]

--example also builds examples/stereonet_infer.cpp (the torch-free whole-model host, include/snb200.h) with the same nvcc flags,
linked against libsnb200.so; OUT defaults to build/stereonet_infer next to this file.  examples/stereonet_adapt.cpp (the torch-free
adaptation host) is built next to it as stereonet_adapt, and examples/stereonet_adapt_dp.cpp (the torch-free multi-GPU data-parallel
host) as stereonet_adapt_dp when NCCL is installed (the nvidia.nccl package that comes with torch; without it that one example is
skipped with a message)."""
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libsnb200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
         "-cudart", "static"]


def sources():
  return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def stale():
  if not os.path.exists(OUT):
    return True
  t = os.path.getmtime(OUT)
  deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(HERE, "..", "include", "*.h"))
  return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
  if not force and not stale():
    return OUT
  objs = []
  os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
  procs = []
  for src in sources():
    obj = os.path.join(HERE, "build", os.path.basename(src)[:-3] + ".o")
    objs.append(obj)
    if (not force) and os.path.exists(obj) and os.path.getmtime(obj) > max(
        [os.path.getmtime(src)] + [os.path.getmtime(h) for h in glob.glob(os.path.join(CSRC, "*.cuh"))]
        + [os.path.getmtime(h) for h in glob.glob(os.path.join(HERE, "..", "include", "*.h"))]):
      continue
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
  for cmd, p in procs:
    out, _ = p.communicate()
    if verbose or p.returncode != 0:
      print(" ".join(cmd))
      print(out)
    if p.returncode != 0:
      raise RuntimeError("nvcc failed for " + cmd[-3])
  cmd = [NVCC, "-shared", "-o", OUT, "-cudart", "static"] + objs
  subprocess.check_call(cmd)
  return OUT


EXAMPLES = os.path.join(HERE, "..", "examples")


def find_nccl():
  """(include dir, library file) of the NCCL that the nvidia.nccl package installs, or None."""
  try:
    import nvidia.nccl
  except ImportError:
    return None
  for d in nvidia.nccl.__path__:
    inc, libs = os.path.join(d, "include"), sorted(glob.glob(os.path.join(d, "lib", "libnccl.so*")))
    if os.path.exists(os.path.join(inc, "nccl.h")) and libs:
      return inc, libs[0]
  return None


def build_example(out=None, name="stereonet_infer"):
  """examples/<name>.cpp -> `out` (default build/<name>), linked against (and with an rpath to) libsnb200.so; stereonet_adapt_dp
  also against NCCL (RuntimeError if find_nccl() finds none)."""
  lib = build()
  out = out or os.path.join(HERE, "build", name)
  os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
  libdir = os.path.dirname(lib)
  cmd = ([NVCC] + FLAGS + ["-I", os.path.join(HERE, "..", "include"), os.path.join(EXAMPLES, name + ".cpp"), "-o", out,
                           "-L" + libdir, "-lsnb200", "-Xlinker", "-rpath=" + libdir])
  if name == "stereonet_adapt_dp":
    nccl = find_nccl()
    if nccl is None:
      raise RuntimeError("stereonet_adapt_dp needs NCCL: no nccl.h / libnccl.so in the nvidia.nccl package")
    inc, so = nccl
    cmd += ["-I", inc, "-Xlinker", "-l:" + os.path.basename(so), "-L" + os.path.dirname(so),
            "-Xlinker", "-rpath=" + os.path.dirname(so)]
  subprocess.check_call(cmd)
  return out


if __name__ == "__main__":
  print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
  if "--example" in sys.argv:
    i = sys.argv.index("--example")
    nxt = sys.argv[i + 1] if i + 1 < len(sys.argv) and not sys.argv[i + 1].startswith("-") else None
    print(build_example(nxt))
    print(build_example(os.path.join(os.path.dirname(os.path.abspath(nxt)), "stereonet_adapt") if nxt else None, "stereonet_adapt"))
    if find_nccl() is None:
      print("stereonet_adapt_dp: skipped (NCCL not found: no nvidia.nccl package with nccl.h and libnccl.so)")
    else:
      print(build_example(os.path.join(os.path.dirname(os.path.abspath(nxt)), "stereonet_adapt_dp") if nxt else None,
                          "stereonet_adapt_dp"))
