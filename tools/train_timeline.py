"""clock64 timeline of one chain-kernel CTA of the trainer. Needs a side build of the library with the
timeline stamps compiled in (the product build has none):

    cd ethz-safe-learning_b200/csrc && make && \
    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC \
         -DSIMBA_TRAIN_TIMELINE -c trainer_f32.cu -o /tmp/trainer_f32_tl.o && \
    nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ../simba_b200/libsimba_b200_tl.so \
         api.o cem_kernels.o rollout_f32.o rollout_tc.o rollout_tc_wide.o trainer.o trainer_tc.o \
         /tmp/trainer_f32_tl.o -ldl
"""
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
os.environ['SIMBA_B200_LIB'] = os.path.join(ROOT, 'ethz-safe-learning_b200', 'simba_b200', 'libsimba_b200_tl.so')
sys.argv = [sys.argv[0], '--steps', '20']
exec(open(os.path.join(ROOT, 'tools', 'profile_train.py')).read())
lib = _lib.load()
buf = (C.c_longlong * 512)()
lib.simba_debug_train_timeline.argtypes = [C.c_void_p]
assert lib.simba_debug_train_timeline(buf) == 0
t0 = buf[0]
print("start->loop %d, loop_end(sum) %d" % (buf[1] - t0, buf[2] - t0))
for it in range(9):
    b = [buf[8 + it * 8 + j] - t0 for j in range(5)]
    print("chunk %d: top %6d issue %5d wait %5d fma %5d epi %5d" % (it, b[0], b[1] - b[0], b[2] - b[1], b[3] - b[2], b[4] - b[3]))
