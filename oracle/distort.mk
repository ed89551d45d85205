# Builds the CPU oracle of the corner undistortion (kernel K7) and of the board pose on undistorted corners as
# oracle/liba3ref_distort.so (test infrastructure; git-ignored).  A library of its own, so the other oracles are untouched.
HERE := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))
CC ?= gcc
CFLAGS ?= -O3 -std=c11 -fPIC -Wall -Wextra -ffp-contract=off -fno-fast-math

all: $(HERE)liba3ref_distort.so

$(HERE)liba3ref_distort.so: $(HERE)a3ref_distort.c $(HERE)a3ref_distort.h $(HERE)a3ref_board.c $(HERE)a3ref_board.h $(HERE)a3ref_pose.c \
                            $(HERE)a3ref_pose.h $(HERE)../aruco3_b200/csrc/k6_board_spec.h $(HERE)../aruco3_b200/csrc/k7_undistort_spec.h
	$(CC) $(CFLAGS) -shared -o $@ $(HERE)a3ref_distort.c $(HERE)a3ref_board.c $(HERE)a3ref_pose.c -lm

clean:
	rm -f $(HERE)liba3ref_distort.so
