#!/bin/sh
# Commit-able SASS listing of the hot kernels (profiles/<tag>_sass_*.txt) from the in-tree library.
set -e
cd "$(dirname "$0")/.."
tag=${1:-r1}
cuobjdump -sass wab_gym_b200/libwab_b200.so > /tmp/wab_all.sass
python - "$tag" <<'PY'
import re, sys
tag = sys.argv[1]
txt = open('/tmp/wab_all.sass').read()
for f in re.split(r'\n\s*Function : ', txt)[1:]:
    name = f.split('\n', 1)[0]
    for key, out in (('wab_step_kernelILb0ELi1ELi24E', 'step_lpe1'), ('wab_step_kernelILb0ELi16E', 'step_lpe16'), ('wab2_turn_kernel', 'v2_turn'),
                     ('wab_step_pipe_kernelILb0ELi8E', 'step_pipe_lpe8'), ('wab_affine1_tc_kernelILi2E', 'policy_forward_tcgen05'), ('wab_affine1_tc_kernelILi3E', 'policy_act_tcgen05'),
                     ('wab2_grid_turn_kernelILb1ELb0E', 'v2_grid_turn'), ('wab_policy_bwd_kernel', 'policy_backward_tcgen05'),
                     ('wab_policy_ppo_bwd_kernel', 'policy_ppo_backward_tcgen05'), ('wab_policy_eval_kernel', 'policy_eval_tcgen05'),
                     ('wab_policy_logits_bwd_kernel', 'policy_logits_backward_tcgen05')):
        if key in name:
            body = 'Function : ' + f
            # keep the instruction text only: drop the hex encodings (and the encoding-only second line of every instruction)
            body = '\n'.join(re.sub(r'\s*/\* 0x[0-9a-f]{16} \*/\s*$', '', ln) for ln in body.split('\n')
                             if not re.match(r'^\s*/\* 0x[0-9a-f]{16} \*/\s*$', ln))
            n = len(re.findall(r'^\s+/\*[0-9a-f]{4,5}\*/', body, flags=re.M))
            ops = {}
            for m in re.finditer(r'^\s+/\*[0-9a-f]{4,5}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)', body, flags=re.M):
                ops[m.group(1)] = ops.get(m.group(1), 0) + 1
            special = ' '.join('%s x%d' % (k, v) for k, v in sorted(ops.items()) if k.startswith(('UTC', 'LDTM', 'STTM', 'SYNCS', 'UTMA', 'REDUX', 'MATCH', 'VOTE', 'SHFL')))
            open('profiles/%s_sass_%s.txt' % (tag, out), 'w').write('# %d SASS instructions (%.1f KB), cuobjdump -sass wab_gym_b200/libwab_b200.so\n# warp / tensor / barrier mnemonics: %s\n' % (n, n * 16 / 1024, special) + body)
            print(out, n, special)
PY
