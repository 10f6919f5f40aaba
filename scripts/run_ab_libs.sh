# same-box A/B of library builds, alternated: LIBS="a.so b.so" ARGS="--envs 32768" [REPS=2] bash scripts/run_ab_libs.sh
# (libraries are looked up in build/, which travels to the GPU box but stays out of git)
L=${LIBDIR:-$PWD/build}
for rep in $(seq ${REPS:-2}); do for lib in $LIBS; do MOOG_B200_LIB=$L/$lib python bench.py --no-clocks --no-cpu $ARGS 2>/dev/null | python -c "
import json,sys;d=json.loads(sys.stdin.read());print('$lib', 'value %.0f e2e %.0f step_only_ms %.3f call_ms %.3f'%(d['value'],d['e2e']['value'],d['roofline']['kernel_ms'],d['roofline']['timed_step_call_ms']))"; done; done
