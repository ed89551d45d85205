/*
 * Constants of the board pose (kernel K6, k6_board.cu) and of its CPU oracle (oracle/a3ref_board.c), in one place so the
 * two cannot drift apart.  Plain C: the oracle includes it too.
 */
#ifndef A3_K6_BOARD_SPEC_H
#define A3_K6_BOARD_SPEC_H

#define A3_K6_MAX_MARKERS 1024   /* markers a board may have */
#define A3_K6_MAX_CODES 8192     /* dictionary size the id -> slot table covers (the largest shipped one has 5 329) */
#define A3_K6_LANES 32           /* point p is summed by lane p % 32, then an xor-shuffle tree 16, 8, 4, 2, 1 */
#define A3_K6_ITERS 10           /* Levenberg-Marquardt iterations per branch */
#define A3_K6_LAMBDA0 1e-3       /* initial damping: (A + lambda * diag(A)) d = -g */
#define A3_K6_LAMBDA_DOWN 0.1    /* factor after a step that lowered the cost */
#define A3_K6_LAMBDA_UP 10.0     /* factor after a step that did not */
#define A3_K6_NO_SLOT 0xffffu    /* id -> slot table entry of an id that is not on the board */

#endif
