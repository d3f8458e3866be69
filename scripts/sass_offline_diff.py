"""The offline MS-TCN layer and Trans-SVNet head kernels compile to the same SASS as in an earlier build.

    python scripts/sass_offline_diff.py <earlier libsurgvid.so, e.g. from scripts/build_prev_lib.sh> <mstcn.o | libsurgvid.so> [...]

The stream path gave these kernels a template parameter (`OfflineTaps` / `StreamTaps`, `OfflineWindow` / `StreamWindow`), and d_k = 64
gave the head kernel another (`trans_head_kernel<DK, Window>`); the offline instantiations and both d_k = 32 head instantiations must not
change.  Instructions are compared with addresses and symbol names stripped.  Needs cuobjdump, no GPU."""
import difflib
import re
import subprocess
import sys


def funcs(path):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
            continue
        if cur and re.search(r"/\*[0-9a-f]{4,}\*/", line):
            ins = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).split(";")[0].strip()
            res[cur].append(re.sub(r"_Z\S+", "SYM", ins))
    return res


# (earlier build, this build): regular expressions, each matching one kernel name.  The earlier side matches both the names from before
# the stream path and those from before the d_k template parameter of the head kernel.
PAIRS = [("mstcn_layer_tc_kernel(EPKf|INS0_11OfflineTaps)", "mstcn_layer_tc_kernelINS0_11OfflineTaps"),
         ("mstcn_layer_kernelILi64ELi1E(EE|NS0_11OfflineTaps)", "mstcn_layer_kernelILi64ELi1ENS0_11OfflineTaps"),
         ("mstcn_layer_kernelILi32ELi1E(EE|NS0_11OfflineTaps)", "mstcn_layer_kernelILi32ELi1ENS0_11OfflineTaps"),
         ("trans_head_kernel(EPKf|INS0_13OfflineWindow)", "trans_head_kernelILi32ENS0_13OfflineWindow"),
         ("trans_head_kernelINS0_12StreamWindow", "trans_head_kernelILi32ENS0_12StreamWindow")]


def main():
    old, new = funcs(sys.argv[1]), {}
    for p in sys.argv[2:]:
        new.update(funcs(p))
    same = True
    for a, b in PAIRS:
        fa, fb = [k for k in old if re.search(a, k)], [k for k in new if re.search(b, k)]
        assert len(fa) == 1 and len(fb) == 1, (a, fa, b, fb)
        A, B = old[fa[0]], new[fb[0]]
        print(f"{b}: {len(A)} vs {len(B)} instructions, identical={A == B}")
        if A != B:
            same = False
            for line in list(difflib.unified_diff(A, B, lineterm=""))[:40]:
                print("   ", line)
    sys.exit(0 if same else 1)


if __name__ == "__main__":
    main()
