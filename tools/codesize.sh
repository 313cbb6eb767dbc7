#!/bin/bash
# per-device-function SASS size of the fused step kernel (instruction-cache budget, see DESIGN.md)
cd "$(dirname "$0")/.."
cuobjdump -elf mujoco_rl_manipulate_unknown_objects_b200/libgripper_sim_b200.so | grep -E "^\s+0x[0-9a-f]+\s+0x[0-9a-f]+\s+0x[0-9a-f]+.*${1:-k_env_step_ls}" \
 | python3 -c "
import sys,re
tot=0
for l in sys.stdin:
    f=l.split(); sz=int(f[2],16); name=f[-1]
    name=re.sub(r'^\\\$_ZN3grs\d+k_\w+?E[A-Za-z0-9_]*?\\\$','',name)
    if sz: print('%7d  %s'%(sz,name[:100])); tot+=sz if not name.startswith('_ZN3grs') or '\$' in f[-1] else 0
"
