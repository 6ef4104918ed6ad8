#!/usr/bin/env python3
"""Per-kernel SASS comparison of two builds of libb200bpe.so (development helper, not used by tests or bench.py).

    python tools/sass_diff.py OLD.so NEW.so

Prints, for every kernel of OLD: identical / differs (with the number of differing instruction lines) / missing in NEW, and
the kernels only NEW has.  Kernels that became templates are compared with the instantiation that is the old kernel (`k_merge_seg` -> `k_merge_seg<false>`, ...).  Used to
show that the kernels which ran on a B200 at commit 551f44c are the same machine code in the current library:

    git archive 551f44c minbpe_b200/csrc include | tar -x -C /tmp/old && (cd /tmp/old/minbpe_b200/csrc && nvcc <flags of build.py> -o /tmp/old.so b200bpe.cu)
    python tools/sass_diff.py /tmp/old.so minbpe_b200/csrc/libb200bpe.so
"""
import re
import subprocess
import sys


def kernels(so):
    txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    out, name, body = {}, None, []
    for ln in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            if name:
                out[name] = body
            name, body = m.group(1), []
        elif name and re.match(r"\s+/\*[0-9a-f]{4}\*/", ln):
            body.append(re.sub(r"/\*[0-9a-f]{4}\*/", "", ln, count=1).strip())     # drop the address column
        elif name and re.match(r"\s+/\* 0x[0-9a-f]{16} \*/", ln):
            body.append(ln.strip())                                                  # second encoding word
    if name:
        out[name] = body
    dem = subprocess.run(["c++filt"] + list(out), capture_output=True, text=True).stdout.splitlines()
    return {re.sub(r"\(.*", "", d).replace("void ", "").replace(" ", ""): out[k] for k, d in zip(out, dem)}


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    alias = {"k_merge_seg": "k_merge_seg<false>", "k_split_apply<false>": "k_split_apply<false,false,0>",
             "k_split_apply<true>": "k_split_apply<true,false,0>", "k_split_reduce": "k_split_reduce<false>",
             "k_enc_insert": "k_enc_insert<false>", "k_enc_count": "k_enc_count<false>", "k_enc_write": "k_enc_write<false>"}    # became templates
    same = diff = gone = 0
    for k in sorted(old):
        k2 = k if k in new else alias.get(k)
        if k2 not in new:
            print(f"missing in NEW   {k}"); gone += 1
        elif old[k] == new[k2]:
            same += 1
        else:
            pairs = [(a, b) for a, b in zip(old[k], new[k2]) if a != b and not a.startswith("/* 0x")]
            n = len(pairs) + abs(len(old[k]) - len(new[k2])) // 2
            # the same instruction stream up to one immediate (e.g. the base offset of dynamic shared memory)?
            imm = {(re.sub(r"0x[0-9a-f]+", "#", a) == re.sub(r"0x[0-9a-f]+", "#", b)) for a, b in pairs}
            note = "  [only immediates differ: " + ", ".join(sorted({f"{x}->{y}" for a, b in pairs for x, y in zip(re.findall(r"0x[0-9a-f]+", a.split("/*")[0]), re.findall(r"0x[0-9a-f]+", b.split("/*")[0])) if x != y})) + "]" \
                if len(old[k]) == len(new[k2]) and imm == {True} else ""
            print(f"DIFFERS          {k}: {n} instructions ({len(old[k]) // 2} -> {len(new[k2]) // 2}){note}"); diff += 1
    only_new = sorted(set(new) - set(old) - set(alias.values()))
    print(f"{same} identical, {diff} differ, {gone} missing; only in NEW: {len(only_new)}")
    for k in only_new:
        print(f"  new            {k}")


if __name__ == "__main__":
    main()
