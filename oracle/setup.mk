# Builds the C restatement of gnark's setupABC (test infrastructure / CPU baseline of the setup) ->
# oracle/_build/liboracle_setup.so.  Same flags as the Makefile beside it; oracle_setup.c includes oracle.c.
CC := gcc
CFLAGS := -O3 -march=x86-64-v3 -fopenmp -fPIC -shared -std=gnu11 -Wall -Wno-unused-function
OUT := _build/liboracle_setup.so

all: $(OUT)

$(OUT): c/oracle_setup.c c/oracle.c c/oracle_groth16.c
	@mkdir -p _build
	$(CC) $(CFLAGS) -o $@ $<

.PHONY: all
