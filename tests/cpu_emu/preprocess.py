"""TEST INFRASTRUCTURE (see cuda_emu.hpp).  Rewrites a CUDA source so that g++ can compile it against cuda_emu.hpp:

  kernel<targs><<<grid, block, smem, stream>>>(args)   ->  emu::launch(emu::LaunchCfg(grid, block, smem, stream), kernel<targs>, args)
  extern __shared__ T name[];                          ->  T* name = (T*)emu::dyn_smem();
  #include <cuda_runtime.h>                            ->  #include "cuda_emu.hpp"

Nothing else is touched: the kernels' bodies are compiled exactly as written.  usage: preprocess.py in.cu out.cpp"""
import re
import sys


def match_back(s, i):
    """s[i-1] == '>': index of the matching '<'"""
    depth = 0
    j = i - 1
    while j >= 0:
        if s[j] == ">":
            depth += 1
        elif s[j] == "<":
            depth -= 1
            if depth == 0:
                return j
        j -= 1
    raise ValueError("unbalanced template arguments before <<<")


def match_paren(s, i):
    """s[i] == '(': index of the matching ')'"""
    depth = 0
    for j in range(i, len(s)):
        if s[j] == "(":
            depth += 1
        elif s[j] == ")":
            depth -= 1
            if depth == 0:
                return j
    raise ValueError("unbalanced launch arguments")


def rewrite_launches(s):
    out = []
    pos = 0
    while True:
        k = s.find("<<<", pos)
        if k < 0:
            out.append(s[pos:])
            return "".join(out)
        # kernel expression: identifier [<...>] immediately before <<<
        e = k
        while s[e - 1].isspace():
            e -= 1
        b = e
        if s[b - 1] == ">":
            b = match_back(s, b)
        while b > 0 and (s[b - 1].isalnum() or s[b - 1] in "_:"):
            b -= 1
        kernel = s[b:e]
        c = s.find(">>>", k)
        cfg = s[k + 3:c]
        p = c + 3
        while s[p].isspace():
            p += 1
        assert s[p] == "(", f"launch of {kernel}: no argument list"
        q = match_paren(s, p)
        args = s[p + 1:q].strip()
        out.append(s[pos:b])
        out.append(f"emu::launch(emu::LaunchCfg({cfg}), {kernel}" + (f", {args})" if args else ")"))
        pos = q + 1


def main(src, dst):
    s = open(src).read()
    s = rewrite_launches(s)
    s = re.sub(r"extern\s+__shared__\s+(\w+)\s+(\w+)\[\];", r"\1* \2 = (\1*)emu::dyn_smem();", s)
    s = s.replace("#include <cuda_runtime.h>", '#include "cuda_emu.hpp"')
    with open(dst, "w") as f:
        f.write(f'#line 1 "{src}"\n' + s)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
