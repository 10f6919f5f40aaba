"""Instruction count of every kernel and out-of-line device function of a library (`cuobjdump -elf`:
the size of each function symbol, 16 bytes per SASS instruction).  `python scripts/sass_sizes.py <lib.so> [filter]`"""
import re, subprocess, sys
out = subprocess.run(['cuobjdump', '-elf', sys.argv[1]], capture_output=True, text=True).stdout
pat = sys.argv[2] if len(sys.argv) > 2 else ''
counts = {}
# symbol table rows: index, value, size, info (0x2 / 0x12 = local / global function), other, section, name
# (the value of a kernel's own symbol prints as a bare 0)
for m in re.finditer(r'^\s*0x[0-9a-f]+\s+(?:0x[0-9a-f]+|0)\s+(0x[0-9a-f]+)\s+0x1?2\s+\S+\s+\S+\s+(\S+)\s*$', out, re.M):
    name = m.group(2)  # out-of-line functions read $<kernel>$<function>
    if pat in name:
        counts[name] = counts.get(name, 0) + int(m.group(1), 16) // 16
for k, v in sorted(counts.items(), key=lambda kv: -kv[1]):
    print('%7d  %s' % (v, k))
