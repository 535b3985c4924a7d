/* memory_arena.h — the reference's bump allocator (include/memory_arena.h), the calls the drop-in
 * layer and oracle/ref_harness.c make.  TEST INFRASTRUCTURE. */
#ifndef REFAPI_MEMORY_ARENA_H
#define REFAPI_MEMORY_ARENA_H
#include <stdbool.h>
#include <stddef.h>

typedef struct MemoryArena { unsigned char *memory; size_t capacity; size_t offset; } MemoryArena;

bool  mem_arena_init(MemoryArena *arena, size_t capacity);
void *mem_arena_alloc(MemoryArena *arena, size_t size, bool zero);
void  mem_arena_reset(MemoryArena *arena);
void  mem_arena_destroy(MemoryArena *arena);
#endif
