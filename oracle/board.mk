# Builds the CPU oracle of the board pose (kernel K6) as oracle/liba3ref_board.so (test infrastructure; git-ignored).
# A library of its own, so liba3ref.so and liba3ref_refine.so are untouched.
HERE := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))
CC ?= gcc
CFLAGS ?= -O3 -std=c11 -fPIC -Wall -Wextra -ffp-contract=off -fno-fast-math

all: $(HERE)liba3ref_board.so

$(HERE)liba3ref_board.so: $(HERE)a3ref_board.c $(HERE)a3ref_board.h $(HERE)a3ref_pose.c $(HERE)a3ref_pose.h \
                          $(HERE)../aruco3_b200/csrc/k6_board_spec.h
	$(CC) $(CFLAGS) -shared -o $@ $(HERE)a3ref_board.c $(HERE)a3ref_pose.c -lm

clean:
	rm -f $(HERE)liba3ref_board.so
