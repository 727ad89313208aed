#!/bin/bash
# Static size of a kernel and the spans of its loops (backward branches), from a cubin compiled without a GPU:
#   bash tools/loop_size.sh [source.cu] [mangled-name substring] [extra nvcc flags...]
# defaults: hwy_highway.cu, highway_step_kernelILi64ELb1.  Writes $HWY_LOOP_SIZE_DIR/kernel.dis (default
# /tmp/hwy_loop_size) for sass_footprint.py.
set -e
SRC=${1:-hwy_highway.cu}; PAT=${2:-highway_step_kernelILi64ELb1}; shift 2 2>/dev/null || true
export OUT=${HWY_LOOP_SIZE_DIR:-/tmp/hwy_loop_size}; mkdir -p "$OUT"
nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false -cubin "$@" \
  -o "$OUT/k.cubin" highwayenv_b200/csrc/$SRC
nvdisasm -g "$OUT/k.cubin" > "$OUT/all.dis"
PAT=$PAT python - <<'P'
import os, re
pat, out = os.environ['PAT'], os.environ['OUT']
L=open(os.path.join(out, 'all.dis')).read().split('\n')
starts=[k for k,l in enumerate(L) if l.startswith('\t.section\t.text.')]
for a,b in zip(starts,starts[1:]+[len(L)]):
    name=L[a].split('.text.')[1].split(',')[0]
    if pat not in name: continue
    open(os.path.join(out, 'kernel.dis'),'w').write('\n'.join(L[a:b]))
    labels={}; ins=[]
    for l in L[a:b]:
        m=re.match(r'(\.L_x_\d+):',l)
        if m: labels[m.group(1)]=None; continue
        m=re.match(r'\s*/\*([0-9a-f]{4,6})\*/\s+(.*?);',l)
        if m:
            addr=int(m.group(1),16); ins.append((addr,m.group(2)))
            for k,v in labels.items():
                if v is None: labels[k]=addr
    spans=[]
    for addr,t in ins:
        m=re.search(r'BRA\S*\s+(?:!?U?P\d+,\s*)?`\((\.L_x_\d+)\)',t)
        if m and labels.get(m.group(1)) is not None and labels[m.group(1)]<addr:
            spans.append((addr-labels[m.group(1)],labels[m.group(1)],addr))
    spans.sort(reverse=True)
    print(name[:70],'total',ins[-1][0]+16,'B; backward spans:',[(s,hex(lo),hex(hi)) for s,lo,hi in spans[:10]])
P
