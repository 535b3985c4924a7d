/* memory_arena.c — a bump allocator behind memory_arena.h, for the drop-in test harness. TEST INFRASTRUCTURE. */
#include "memory_arena.h"

#include <stdlib.h>
#include <string.h>

bool mem_arena_init(MemoryArena *arena, size_t capacity)
{
    arena->memory = (unsigned char *)malloc(capacity);
    arena->capacity = arena->memory ? capacity : 0;
    arena->offset = 0;
    return arena->memory != NULL;
}

void *mem_arena_alloc(MemoryArena *arena, size_t size, bool zero)
{
    size_t start = (arena->offset + 63) & ~(size_t)63;
    if (!arena->memory || start > arena->capacity || size > arena->capacity - start) return NULL;
    arena->offset = start + size;
    if (zero) memset(arena->memory + start, 0, size);
    return arena->memory + start;
}

void mem_arena_reset(MemoryArena *arena) { arena->offset = 0; }

void mem_arena_destroy(MemoryArena *arena)
{
    free(arena->memory);
    arena->memory = NULL;
    arena->capacity = arena->offset = 0;
}
