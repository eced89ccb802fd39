# oracle/ksw.mk -- builds the test-only CPU restatement of BWA-MEM's seed extension (ksw_oracle.c, bwa's ksw_extend2)
# as its own library, libksw_oracle.so (integer arithmetic only: no floating-point flags to pin).
CC ?= gcc

all: libksw_oracle.so

libksw_oracle.so: ksw_oracle.c
	$(CC) -O2 -std=gnu11 -fPIC -shared -o $@ ksw_oracle.c

clean:
	rm -f libksw_oracle.so

.PHONY: all clean
