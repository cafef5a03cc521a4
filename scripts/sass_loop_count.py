"""Instruction classes of one loop body in `cuobjdump -sass` output.

usage: sass_loop_count.py <file.sass> <first_hex> <last_hex>
counts the instructions at addresses first..last (inclusive; e.g. a loop's back-branch target and the back-branch
itself) by class: packed FP32 (FFMA2/FMUL2/FADD2), scalar FP32, compare/select/logic (ALU pipe), SHFL, LDS, STS,
MUFU and the rest.
"""
import collections
import re
import sys

CLASSES = {
    "FP32x2": ["FFMA2", "FMUL2", "FADD2"],
    "FP32": ["FFMA", "FMUL", "FADD"],
    "ALU": ["FSETP", "FSEL", "SEL", "FMNMX", "ISETP", "LOP3", "PLOP3", "SHF", "LEA", "IMNMX"],
    "SHFL": ["SHFL"],
    "LDS": ["LDS"],
    "STS": ["STS"],
    "MUFU": ["MUFU"],
}


def main():
    path, first, last = sys.argv[1], int(sys.argv[2], 16), int(sys.argv[3], 16)
    ops = collections.Counter()
    for line in open(path):
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z0-9_]+)", line)
        if m and first <= int(m.group(1), 16) <= last:
            ops[m.group(3)] += 1
    print("total", sum(ops.values()))
    rest = dict(ops)
    for name, members in CLASSES.items():
        print(name, sum(ops[o] for o in members), {o: ops[o] for o in members if ops[o]})
        for o in members:
            rest.pop(o, None)
    print("other", sum(rest.values()), rest)


if __name__ == "__main__":
    main()
