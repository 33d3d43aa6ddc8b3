"""Build libmobody_b200 with extra -D flags into variants/<name>/ (A/B experiments on the GPU box).

usage: python scripts/build_variant.py NAME -DUG_TRACE ...   ->  variants/NAME/libmobody_b200.so
Select it at run time with MOBODY_B200_LIB=variants/NAME/libmobody_b200.so.
"""
import os, subprocess, sys
from concurrent.futures import ThreadPoolExecutor
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mobody_b200 import build as B

name, flags = sys.argv[1], sys.argv[2:]
out = os.path.join(ROOT, "variants", name)
os.makedirs(out, exist_ok=True)

def cc(src):
    obj = os.path.join(out, src.replace(".cu", ".o"))
    subprocess.run([B._nvcc()] + B.NVCC_FLAGS + flags + ["-c", os.path.join(B.CSRC, src), "-o", obj], check=True)
    return obj

with ThreadPoolExecutor(8) as ex:
    objs = list(ex.map(cc, B.SOURCES))
lib = os.path.join(out, "libmobody_b200.so")
subprocess.run([B._nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs + ["-lcudart"], check=True)
for o in objs:
    os.remove(o)
print(lib)
