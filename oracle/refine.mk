# Builds the CPU oracle of the corner refinement (kernel K5) and its f32-corner pose entries as oracle/liba3ref_refine.so
# (test infrastructure; git-ignored).  A library of its own, so the parity oracle (Makefile, liba3ref.so) is untouched.
HERE := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))
CC ?= gcc
CFLAGS ?= -O3 -std=c11 -fPIC -Wall -Wextra -ffp-contract=off -fno-fast-math

all: $(HERE)liba3ref_refine.so

$(HERE)liba3ref_refine.so: $(HERE)a3ref_refine.c $(HERE)a3ref_refine.h $(HERE)a3ref_pose.c $(HERE)a3ref_pose.h \
                           $(HERE)../aruco3_b200/csrc/k5_refine_spec.h
	$(CC) $(CFLAGS) -shared -o $@ $(HERE)a3ref_refine.c $(HERE)a3ref_pose.c -lm

clean:
	rm -f $(HERE)liba3ref_refine.so
