import re,sys
cur=None
for line in open(sys.argv[1]):
    m=re.search(r"Function properties for (\S+)",line)
    if m: cur=m.group(1)
    m=re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads",line)
    if m and cur and "conv_umma" in cur: sp=m.groups()
    m=re.search(r"Used (\d+) registers",line)
    if m and cur and "conv_umma" in cur:
        t=re.search(r"k_conv_umma(I.*)EEvNS0",cur); print(t.group(1) if t else cur, "regs",m.group(1),"spill st/ld",sp); cur=None
