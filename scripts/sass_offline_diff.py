"""Kernels compile to the same SASS as in an earlier build.  Needs cuobjdump, no GPU.

    python scripts/sass_offline_diff.py <earlier libsurgvid.so, e.g. from scripts/build_prev_lib.sh> <mstcn.o | libsurgvid.so> [...]
    python scripts/sass_offline_diff.py --all <earlier libsurgvid.so> <libsurgvid.so> [...]

Default: the offline MS-TCN layer and Trans-SVNet head kernels, and the LayerNorm kernel.  The stream path gave these kernels a
template parameter (`OfflineTaps` / `StreamTaps`, `OfflineWindow` / `StreamWindow`), and d_k = 64 gave the head kernel another
(`trans_head_kernel<DK, Window>`); the offline instantiations and both d_k = 32 head instantiations must not change.  The channel-major
output form gave `layernorm_kernel<LPR, NV, EXACT, NCHW>` its last parameter; the 32 token-major instantiations must not change.

--all: every kernel of the two builds, matched by name, for changes that must not touch device code (host-only refactors).  Both builds
must have the same set of kernels.  Names in an anonymous namespace carry per-file hashes (`_GLOBAL__N__<8 hex>`, `_cu_<8 hex>`) that
change with any edit of the file; they are replaced by a placeholder before matching.  ptxas output also depends on the address-space
layout of the compiling process (two builds of the same source can allocate registers differently), so build both libraries with address
randomisation off, e.g. `setarch "$(uname -m)" -R scripts/build_prev_lib.sh <commit>` and the same around the current build.

Instructions are compared with addresses and symbol names stripped."""
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


# (earlier build, this build): regular expressions, each matching one kernel name.  The earlier side matches the names from before the
# stream path, those from before the d_k template parameter of the head kernel, and the current ones.
PAIRS = [("mstcn_layer_tc_kernel(EPKf|INS0_11OfflineTaps)", "mstcn_layer_tc_kernelINS0_11OfflineTaps"),
         ("mstcn_layer_kernelILi64ELi1E(EE|NS0_11OfflineTaps)", "mstcn_layer_kernelILi64ELi1ENS0_11OfflineTaps"),
         ("mstcn_layer_kernelILi32ELi1E(EE|NS0_11OfflineTaps)", "mstcn_layer_kernelILi32ELi1ENS0_11OfflineTaps"),
         ("trans_head_kernel(EPKf|INS0_13OfflineWindow|ILi32ENS0_13OfflineWindow)", "trans_head_kernelILi32ENS0_13OfflineWindow"),
         ("trans_head_kernel(INS0_12StreamWindow|ILi32ENS0_12StreamWindow)", "trans_head_kernelILi32ENS0_12StreamWindow")]
# the lane mappings of the LayerNorm dispatch table (elementwise.cu), exact and predicated; the earlier name has no NCHW parameter
PAIRS += [(f"layernorm_kernelILi{l}ELi{n}ELb{e}EEEv", f"layernorm_kernelILi{l}ELi{n}ELb{e}ELb0EEEv")
          for l, n in ((2, 2), (4, 2), (8, 2), (8, 4), (16, 4), (32, 4), (2, 5), (4, 5), (8, 5), (16, 5), (4, 1), (8, 1), (16, 1), (32, 1),
                       (32, 2), (32, 3)) for e in (0, 1)]


def by_stable_name(res):
    out = {}
    for name, ins in res.items():
        key = re.sub(r"_cu_[0-9a-f]{8}", "_cu_H", re.sub(r"_GLOBAL__N__[0-9a-f]{8}", "_GLOBAL__N__H", name))
        assert key not in out, key
        out[key] = ins
    return out


def compare(name, A, B):
    print(f"{name}: {len(A)} vs {len(B)} instructions, identical={A == B}")
    if A != B:
        for line in list(difflib.unified_diff(A, B, lineterm=""))[:40]:
            print("   ", line)
    return A == B


def main():
    every = sys.argv[1] == "--all"
    args = sys.argv[2:] if every else sys.argv[1:]
    old, new = funcs(args[0]), {}
    for p in args[1:]:
        new.update(funcs(p))
    same = True
    if every:
        old, new = by_stable_name(old), by_stable_name(new)
        for k in sorted(old.keys() ^ new.keys()):
            print(f"only in {'the earlier' if k in old else 'this'} build: {k}")
            same = False
        for k in sorted(old.keys() & new.keys()):
            same = compare(k, old[k], new[k]) and same
        print(f"{len(old.keys() & new.keys())} kernels in both builds, all identical={same}")
    else:
        for a, b in PAIRS:
            fa, fb = [k for k in old if re.search(a, k)], [k for k in new if re.search(b, k)]
            assert len(fa) == 1 and len(fb) == 1, (a, fa, b, fb)
            same = compare(b, old[fa[0]], new[fb[0]]) and same
    sys.exit(0 if same else 1)


if __name__ == "__main__":
    main()
